"""Host-side mirror (Python) of the libsdr node interface for the hot path.

Same names, constructor arguments, config()/process() meaning and error behaviour as
  IQBaseBand<Scalar>      src/baseband.hh:21-297
  FMDemod<iScalar,oScalar> src/demod.hh:172-266
  AMDemod / USBDemod      src/demod.hh:16-166
on top of the C ABI (include/sdrg.h).  Arrays are numpy (host entry points) or torch CUDA tensors
(device entry points, asynchronous on the current torch stream).  The C++ mirror of the same
interface (sdr::Sink<T>/Source/Buffer<T>) is include/sdrg/*.hh.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import (Config, ConfigError, T_S8, T_S16, T_F32, T_CS8, T_CS16, T_CF32,  # noqa: F401
                   DEMOD_NONE, DEMOD_FM, DEMOD_AM, DEMOD_USB)

_SCALARS = {"s8": T_S8, "s16": T_S16, "f32": T_F32, np.int8: T_S8, np.int16: T_S16, np.float32: T_F32,
            T_S8: T_S8, T_S16: T_S16, T_F32: T_F32}
_NP = {T_S8: np.int8, T_S16: np.int16, T_F32: np.float32}
_CTYPE = {T_S8: T_CS8, T_S16: T_CS16, T_F32: T_CF32}


def scalar_id(s):
    if isinstance(s, np.dtype):
        s = s.type
    return _SCALARS[s]


def _np_ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev_in(x, dtype=None, what="input"):
    """A torch tensor handed to a *_dev entry point: it must live on a GPU, be contiguous (the C ABI sees a raw
    pointer and a length) and have the element type the node was built for.  Raises ConfigError otherwise --
    a wrong dtype or a strided view would otherwise be read as garbage or past the end."""
    import torch
    if not x.is_cuda:
        raise ConfigError("%s tensor must live on a CUDA device" % what)
    if not x.is_contiguous():
        raise ConfigError("%s tensor must be contiguous (call .contiguous())" % what)
    if dtype is not None:
        want = {np.int8: (torch.int8,), np.uint8: (torch.uint8,), np.int16: (torch.int16,), np.float32: (torch.float32, torch.complex64),
                np.complex64: (torch.complex64, torch.float32)}[np.dtype(dtype).type]
        if x.dtype not in want:
            raise ConfigError("%s tensor has dtype %s, the node expects %s" % (what, x.dtype, np.dtype(dtype).name))
    return C.c_void_p(x.data_ptr())


def fm_out_dtype(scalar):
    return np.float32 if scalar == T_F32 else np.int16


class IQBaseBand:
    """IQBaseBand<Scalar>(Fc, Ff, width, order, sub_sample, oFs=0)  (src/baseband.hh:47-57).
    The 5-argument reference constructor (Ff = Fc, baseband.hh:35) is `IQBaseBand(scalar, Fc, None, ...)`."""

    _in_shape = (-1, 2)

    def __init__(self, scalar, Fc, Ff, width, order, sub_sample, oFs=0.0):
        self.scalar = scalar_id(scalar)
        self.dtype = _NP[self.scalar]
        self._h = C.c_void_p()
        if Ff is None:
            Ff = Fc
        _lib.call("sdrg_iqbb_create", self.scalar, float(Fc), float(Ff), float(width), int(order),
                  int(sub_sample), float(oFs), C.byref(self._h))
        self.out_config = Config()

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.load().sdrg_iqbb_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # setters (baseband.hh:69-112)
    def setCenterFrequency(self, Fc): _lib.call("sdrg_iqbb_set_center_frequency", self._h, float(Fc))
    def setFilterFrequency(self, Ff): _lib.call("sdrg_iqbb_set_filter_frequency", self._h, float(Ff))
    def setFilterWidth(self, w): _lib.call("sdrg_iqbb_set_filter_width", self._h, float(w))
    def setOrder(self, o): _lib.call("sdrg_iqbb_set_order", self._h, int(o))
    def setSubsample(self, ss): _lib.call("sdrg_iqbb_set_subsample", self._h, int(ss))
    def setOutputSampleRate(self, fs): _lib.call("sdrg_iqbb_set_output_sample_rate", self._h, float(fs))

    def setInputType(self, type_id):
        """int16 only: consume complex uint8 / int8 input with AutoCast<complex<int16>> fused into the load."""
        _lib.call("sdrg_iqbb_set_input_type", self._h, int(type_id))
        self.in_dtype = {_lib.T_CU8: np.uint8, _lib.T_CS8: np.int8}.get(int(type_id), self.dtype)
        self._in_type = int(type_id)

    def setFloatPath(self, mode):
        """f32 only: 0 auto, 1 direct kernel, 2 folded kernel (before config())."""
        _lib.call("sdrg_iqbb_set_float_path", self._h, int(mode))

    def lastFloatKernel(self):
        """Diagnostics: 1 direct FIR, 2 folded batched, 3 window-pipelined, 4 staged short windows, 5 per-window."""
        w = C.c_int(0)
        _lib.call("sdrg_iqbb_last_float_kernel", self._h, C.byref(w))
        return w.value

    def config(self, src_cfg=None, *, type=None, sample_rate=0.0, buffer_size=0, num_buffers=1):
        """config(const Config&) (baseband.hh:115-132). Raises ConfigError on a type mismatch."""
        if src_cfg is None:
            src_cfg = Config(self._ctype() if type is None else type, sample_rate, buffer_size, num_buffers)
        out = Config()
        _lib.call("sdrg_iqbb_configure", self._h, C.byref(src_cfg), C.byref(out))
        self.out_config = out
        return out

    def design_only(self, src_cfg=None, *, type=None, sample_rate=0.0, buffer_size=0, num_buffers=1):
        """Host half of config() (no device needed); the node stays unconfigured for process()."""
        if src_cfg is None:
            src_cfg = Config(self._ctype() if type is None else type, sample_rate, buffer_size, num_buffers)
        out = Config()
        _lib.call("sdrg_iqbb_design", self._h, C.byref(src_cfg), C.byref(out))
        self.out_config = out
        return out

    def _ctype(self):
        return getattr(self, "_in_type", _CTYPE[self.scalar])

    def info(self):
        inf = _lib.IqbbInfo()
        _lib.call("sdrg_iqbb_get_info", self._h, C.byref(inf), None, None)
        return inf

    def design(self):
        """(kernel, lut) exactly as the node uses them: int32 pairs, or float32 pairs for f32."""
        inf = self.info()
        dt = np.float32 if self.scalar == T_F32 else np.int32
        k = np.zeros((inf.order, 2), dtype=dt); lut = np.zeros((128, 2), dtype=dt)
        _lib.call("sdrg_iqbb_get_info", self._h, C.byref(inf), _np_ptr(k), _np_ptr(lut))
        return k, lut

    def outputs_for(self, n_in):
        n = C.c_size_t(0)
        _lib.call("sdrg_iqbb_outputs_for", self._h, int(n_in), C.byref(n))
        return n.value

    def process(self, x):
        """process(buffer): returns the outputs this buffer completes (baseband.hh:136-223)."""
        if _is_torch(x):
            import torch
            n_in = x.shape[0]
            n_out = self.outputs_for(n_in)
            odt = {np.int8: torch.int8, np.int16: torch.int16, np.float32: torch.float32}[self.dtype]
            out = torch.empty((max(n_out, 1), 2), dtype=odt, device=x.device)
            got = C.c_size_t(0)
            _lib.call("sdrg_iqbb_process_dev", self._h, _dev_in(x, getattr(self, "in_dtype", self.dtype)), n_in,
                      C.c_void_p(out.data_ptr()), n_out, C.byref(got), _stream_ptr())
            return out[:got.value]
        x = np.ascontiguousarray(x, dtype=getattr(self, "in_dtype", self.dtype)).reshape(self._in_shape)
        n_out = self.outputs_for(x.shape[0])
        out = np.zeros((n_out, 2), dtype=self.dtype)
        got = C.c_size_t(0)
        _lib.call("sdrg_iqbb_process", self._h, _np_ptr(x), x.shape[0], _np_ptr(out), n_out, C.byref(got))
        return out[:got.value]


class BaseBand(IQBaseBand):
    """BaseBand<Scalar>(Fc, Ff, width, order, sub_sample) on a REAL stream (src/baseband.hh:304-529), Scalar = int16_t
    (default) or int8_t: complex band-pass FIR (gain 2^16 resp. 2^8) -> NCO -> mean of exactly sub_sample samples;
    output (n, 2) of the same scalar.  The int8 instantiation computes in 16 bits throughout, like the reference.
    The 4-argument reference constructor (Ff = Fc, baseband.hh:322) is `BaseBand(Fc, None, ...)`."""

    _in_shape = (-1,)

    def __init__(self, Fc, Ff, width, order, sub_sample, scalar="s16"):
        self.scalar = scalar_id(scalar)
        self.dtype = _NP[self.scalar]
        self._in_type = self.scalar
        self._h = C.c_void_p()
        if Ff is None:
            Ff = Fc
        _lib.call("sdrg_iqbb_create_real", self.scalar, float(Fc), float(Ff), float(width), int(order),
                  int(sub_sample), C.byref(self._h))
        self.out_config = Config()

    def setFrequencyShift(self, Fc):
        """FreqShiftBase::setFrequencyShift (src/freqshift.hh:62-65)."""
        _lib.call("sdrg_iqbb_set_center_frequency", self._h, float(Fc))


class FMDemod:
    """FMDemod<iScalar, oScalar> (src/demod.hh:172-266); int input -> int16, float -> float."""

    def __init__(self, scalar):
        self.scalar = scalar_id(scalar)
        self._h = C.c_void_p()
        _lib.call("sdrg_fmdemod_create", self.scalar, C.byref(self._h))

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.load().sdrg_fmdemod_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def config(self, src_cfg):
        out = Config()
        _lib.call("sdrg_fmdemod_configure", self._h, C.byref(src_cfg), C.byref(out))
        return out

    def process(self, x, in_place=True, out=None):
        """Element 0 is skipped like the reference: in_place -> the aliased input bytes, else `out[0]`
        (or 0 when no `out` array is passed) is left untouched."""
        if _is_torch(x):
            import torch
            n = x.shape[0]
            odt = torch.float32 if self.scalar == T_F32 else torch.int16
            if out is None:
                out = torch.zeros(max(n, 1), dtype=odt, device=x.device)
            _lib.call("sdrg_fmdemod_process_dev", self._h, _dev_in(x, _NP[self.scalar]), n,
                      C.c_void_p(out.data_ptr()), int(in_place), _stream_ptr())
            return out[:n]
        x = np.ascontiguousarray(x, dtype=_NP[self.scalar]).reshape(-1, 2)
        n = x.shape[0]
        if out is None:
            out = np.zeros(n, dtype=fm_out_dtype(self.scalar))
        _lib.call("sdrg_fmdemod_process", self._h, _np_ptr(x), n, _np_ptr(out), int(in_place))
        return out


class _Envelope:
    _name = ""

    def __init__(self, scalar):
        self.scalar = scalar_id(scalar)

    def config(self, src_cfg):
        out = Config()
        _lib.call("sdrg_%s_configure" % self._name, self.scalar, C.byref(src_cfg), C.byref(out))
        return out

    def process(self, x):
        if _is_torch(x):
            import torch
            n = x.shape[0]
            out = torch.empty(max(n, 1), dtype=x.dtype, device=x.device)
            _lib.call("sdrg_%s_process_dev" % self._name, self.scalar, _dev_in(x, _NP[self.scalar]), n,
                      C.c_void_p(out.data_ptr()), _stream_ptr())
            return out[:n]
        x = np.ascontiguousarray(x, dtype=_NP[self.scalar]).reshape(-1, 2)
        out = np.zeros(x.shape[0], dtype=_NP[self.scalar])
        _lib.call("sdrg_%s_process" % self._name, self.scalar, _np_ptr(x), x.shape[0], _np_ptr(out))
        return out


class AMDemod(_Envelope):
    """AMDemod<Scalar> (src/demod.hh:16-86)."""
    _name = "amdemod"


class USBDemod(_Envelope):
    """USBDemod<Scalar> (src/demod.hh:91-166)."""
    _name = "usbdemod"


class RxChain:
    """IQBaseBand -> demod over many buffers per launch (sdrg_rxchain_*): the equivalent of
    n_buffers Source::send() calls through directly connected, in-place nodes."""

    def __init__(self, baseband, demod):
        self.bb = baseband
        self.demod = demod
        self._h = C.c_void_p()
        _lib.call("sdrg_rxchain_create", baseband._h, int(demod), C.byref(self._h))

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.load().sdrg_rxchain_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def reset(self):
        _lib.call("sdrg_rxchain_reset", self._h)

    def audio_dtype(self):
        if self.demod == DEMOD_FM:
            return fm_out_dtype(self.bb.scalar)
        return self.bb.dtype

    def process(self, x, buffer_size, bb_out=None, audio_out=None):
        """x: (n_buffers*buffer_size, 2). Returns (bb, audio, counts)."""
        n_total = x.shape[0]
        assert n_total % buffer_size == 0
        nb = n_total // buffer_size
        n_out = self.bb.outputs_for(n_total)
        counts = (C.c_size_t * nb)()
        got = C.c_size_t(0)
        if _is_torch(x):
            import torch
            adt = {np.int16: torch.int16, np.int8: torch.int8, np.float32: torch.float32}[self.audio_dtype()]
            if bb_out is None:
                bdt = {np.int16: torch.int16, np.int8: torch.int8, np.float32: torch.float32}[self.bb.dtype]
                bb_out = torch.empty((max(n_out, 1), 2), dtype=bdt, device=x.device)
            if audio_out is None:
                audio_out = torch.zeros(max(n_out, 1), dtype=adt, device=x.device)
            _lib.call("sdrg_rxchain_process_dev", self._h, _dev_in(x, getattr(self.bb, "in_dtype", self.bb.dtype)), buffer_size, nb,
                      _dev_in(bb_out, self.bb.dtype, "bb_out"), _dev_in(audio_out, self.audio_dtype(), "audio_out"), n_out,
                      C.byref(got), counts, _stream_ptr())
            return bb_out[:got.value], audio_out[:got.value], np.array(counts[:], dtype=np.int64)
        x = np.ascontiguousarray(x, dtype=getattr(self.bb, "in_dtype", self.bb.dtype)).reshape(-1, 2)
        if bb_out is None:
            bb_out = np.zeros((n_out, 2), dtype=self.bb.dtype)
        if audio_out is None:
            audio_out = np.zeros(n_out, dtype=self.audio_dtype())
        _lib.call("sdrg_rxchain_process", self._h, _np_ptr(x), buffer_size, nb, _np_ptr(bb_out),
                  _np_ptr(audio_out), n_out, C.byref(got), counts)
        return bb_out[:got.value], audio_out[:got.value], np.array(counts[:], dtype=np.int64)


    def process_into(self, x, buffer_size, bb_ptr, audio_ptr, out_cap):
        """Device entry point with raw output addresses (e.g. inside a PeerWindow on another GPU):
        bb_ptr / audio_ptr are integers or None.  Returns the number of outputs."""
        nb = x.shape[0] // buffer_size
        got = C.c_size_t(0)
        _lib.call("sdrg_rxchain_process_dev", self._h, _dev_in(x, getattr(self.bb, "in_dtype", self.bb.dtype)), buffer_size, nb,
                  C.c_void_p(bb_ptr) if bb_ptr else None, C.c_void_p(audio_ptr) if audio_ptr else None,
                  int(out_cap), C.byref(got), None, _stream_ptr())
        return got.value


class FFTPlan:
    """FFTPlan<float> (src/fftplan_fftw3.hh:79-142): FFTPlan(n, direction) with direction FORWARD/BACKWARD;
    calling the plan transforms `batch` contiguous n-point signals (complex64)."""
    FORWARD, BACKWARD = 0, 1

    def __init__(self, n, direction):
        self.n = int(n)
        self._h = C.c_void_p()
        _lib.call("sdrg_fft_create", self.n, int(direction), C.byref(self._h))

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.load().sdrg_fft_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def __call__(self, x):
        if _is_torch(x):
            import torch
            out = torch.empty_like(x)
            _lib.call("sdrg_fft_exec_dev", self._h, _dev_in(x, np.complex64), C.c_void_p(out.data_ptr()),
                      x.numel() // self.n, _stream_ptr())
            return out
        x = np.ascontiguousarray(x, dtype=np.complex64)
        out = np.empty_like(x)
        _lib.call("sdrg_fft_exec", self._h, _np_ptr(x), _np_ptr(out), x.size // self.n)
        return out


class FFTPlan64:
    """FFTPlan<double> (src/fftplan_fftw3.hh:12-75): complex128 in / out, any size."""
    FORWARD, BACKWARD = 0, 1

    def __init__(self, n, direction):
        self.n = int(n)
        self._h = C.c_void_p()
        _lib.call("sdrg_fft64_create", self.n, int(direction), C.byref(self._h))

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.load().sdrg_fft64_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def __call__(self, x):
        x = np.ascontiguousarray(x, dtype=np.complex128)
        out = np.empty_like(x)
        _lib.call("sdrg_fft64_exec", self._h, _np_ptr(x), _np_ptr(out), x.size // self.n)
        return out


class FilterNode:
    """FilterNode<float>(block_size) (src/filternode.hh:231-283): addFilter(fmin, fmax) returns the
    filter's index; process(x) returns an array (n_filters, n_out) of complex64."""

    def __init__(self, block_size=1024):
        self.block = int(block_size)
        self._h = C.c_void_p()
        _lib.call("sdrg_filter_create", self.block, C.byref(self._h))

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.load().sdrg_filter_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def addFilter(self, fmin, fmax):
        idx = C.c_size_t(0)
        _lib.call("sdrg_filter_add", self._h, float(fmin), float(fmax), C.byref(idx))
        return idx.value

    def setFreq(self, index, fmin, fmax):
        _lib.call("sdrg_filter_set_freq", self._h, int(index), float(fmin), float(fmax))

    def n_filters(self):
        n = C.c_size_t(0)
        _lib.call("sdrg_filter_count", self._h, C.byref(n))
        return n.value

    def config(self, src_cfg=None, *, sample_rate=0.0, buffer_size=0, num_buffers=1, type=T_CF32):
        if src_cfg is None:
            src_cfg = Config(type, sample_rate, buffer_size, num_buffers)
        out = Config()
        _lib.call("sdrg_filter_configure", self._h, C.byref(src_cfg), C.byref(out))
        return out

    def design(self, index):
        kern = np.zeros(2 * self.block, dtype=np.complex64); taps = np.zeros(self.block, dtype=np.complex64)
        _lib.call("sdrg_filter_get_design", self._h, int(index), _np_ptr(kern), _np_ptr(taps))
        return kern, taps

    def outputs_for(self, n_in):
        n = C.c_size_t(0)
        _lib.call("sdrg_filter_outputs_for", self._h, int(n_in), C.byref(n))
        return n.value

    def process(self, x):
        """Without filters the stream still advances (history, pending samples), and the result has no rows, like a
        FilterSink without sources."""
        F = self.n_filters()
        got = C.c_size_t(0)
        if _is_torch(x):
            import torch
            n_in = x.shape[0]
            n_out = self.outputs_for(n_in)
            out = torch.empty((max(F, 1), max(n_out, 1)), dtype=torch.complex64, device=x.device)
            _lib.call("sdrg_filter_process_dev", self._h, _dev_in(x, np.complex64), n_in, C.c_void_p(out.data_ptr()),
                      max(n_out, 1), C.byref(got), _stream_ptr())
            return out[:F, :got.value]
        x = np.ascontiguousarray(x, dtype=np.complex64).reshape(-1)
        n_out = self.outputs_for(x.shape[0])
        out = np.zeros((max(F, 1), max(n_out, 1)), dtype=np.complex64)
        _lib.call("sdrg_filter_process", self._h, _np_ptr(x), x.shape[0], _np_ptr(out), max(n_out, 1), C.byref(got))
        return out[:F, :got.value]


class ChannelBank:
    """C independent IQBaseBand<Scalar>(Fc[c], Ff[c], width, order, sub_sample, oFs) nodes on one input
    stream, each with FM/AM/USB demodulators connected out of place (sdrg_bank_*).  Scalar "s8" / "s16"
    (bit-exact), or "f32": complex float input, float outputs (FM float32, as fm_out_dtype)."""

    _in_shape = (-1, 2)
    _prefix = "sdrg_bank"

    def __init__(self, scalar, Fc, Ff, width, order, sub_sample, oFs=0.0):
        self.scalar = scalar_id(scalar)
        self.dtype = _NP[self.scalar]
        Fc = np.ascontiguousarray(Fc, dtype=np.float64)
        Ff = Fc if Ff is None else np.ascontiguousarray(Ff, dtype=np.float64)
        self.channels = Fc.shape[0]
        self._h = C.c_void_p()
        dp = C.POINTER(C.c_double)
        _lib.call("sdrg_bank_create", self.scalar, self.channels, Fc.ctypes.data_as(dp), Ff.ctypes.data_as(dp),
                  float(width), int(order), int(sub_sample), float(oFs), C.byref(self._h))

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.load().sdrg_bank_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def config(self, src_cfg=None, *, sample_rate=0.0, buffer_size=0, num_buffers=1, type=None):
        if src_cfg is None:
            src_cfg = Config(_CTYPE[self.scalar] if type is None else type, sample_rate, buffer_size, num_buffers)
        out = Config()
        _lib.call(self._prefix + "_configure", self._h, C.byref(src_cfg), C.byref(out))
        return out

    def outputs_for(self, n_in):
        n = C.c_size_t(0)
        _lib.call(self._prefix + "_outputs_for", self._h, int(n_in), C.byref(n))
        return n.value

    def channel_info(self, c):
        inf = _lib.IqbbInfo()
        k = np.zeros((1024, 2), dtype=np.float32 if self.scalar == T_F32 else np.int32)
        _lib.call("sdrg_bank_get_info", self._h, None, None, int(c), C.byref(inf), _np_ptr(k))
        return inf, k[:inf.order]

    def process(self, x, buffer_size, want=("bb", "fm", "am", "usb"), out=None):
        """x: (n_buffers*buffer_size, 2). Returns dict name -> (channels, n_out) array/tensor."""
        n_total = x.shape[0]
        assert n_total % buffer_size == 0
        nb = n_total // buffer_size
        n_out = self.outputs_for(n_total)
        stride = max(n_out, 1)
        got = C.c_size_t(0)
        res = {} if out is None else out
        if _is_torch(x):
            import torch
            tdt = {np.int16: torch.int16, np.int8: torch.int8, np.float32: torch.float32}[self.dtype]
            fdt = {np.int16: torch.int16, np.float32: torch.float32}[fm_out_dtype(self.scalar)]
            shapes = {"bb": ((self.channels, stride, 2), tdt), "fm": ((self.channels, stride), fdt),
                      "am": ((self.channels, stride), tdt), "usb": ((self.channels, stride), tdt)}
            for k in want:
                if k not in res:
                    res[k] = torch.zeros(shapes[k][0], dtype=shapes[k][1], device=x.device)
            stride = res[want[0]].shape[1]
            ptr = lambda k: C.c_void_p(res[k].data_ptr()) if k in want else None  # noqa: E731
            _lib.call(self._prefix + "_process_dev", self._h, _dev_in(x, self.dtype), buffer_size, nb, ptr("bb"), ptr("fm"),
                      ptr("am"), ptr("usb"), stride, C.byref(got), _stream_ptr())
            return {k: res[k][:, :got.value] for k in want}
        x = np.ascontiguousarray(x, dtype=self.dtype).reshape(-1, 2)
        shapes = {"bb": ((self.channels, stride, 2), self.dtype), "fm": ((self.channels, stride), fm_out_dtype(self.scalar)),
                  "am": ((self.channels, stride), self.dtype), "usb": ((self.channels, stride), self.dtype)}
        for k in want:
            if k not in res:
                res[k] = np.zeros(shapes[k][0], dtype=shapes[k][1])
        ptr = lambda k: _np_ptr(res[k]) if k in want else None  # noqa: E731
        _lib.call(self._prefix + "_process", self._h, _np_ptr(x), buffer_size, nb, ptr("bb"), ptr("fm"), ptr("am"), ptr("usb"),
                  stride, C.byref(got))
        return {k: res[k][:, :got.value] for k in want}


def _bank_process_into(self, x, buffer_size, ptrs, stride):
    """Device entry point with raw output addresses: ptrs maps "bb"/"fm"/"am"/"usb" to integer device
    addresses of (channels, stride) arrays (e.g. rows of a PeerWindow on another GPU)."""
    nb = x.shape[0] // buffer_size
    got = C.c_size_t(0)
    p = lambda k: C.c_void_p(ptrs[k]) if ptrs.get(k) else None  # noqa: E731
    _lib.call(self._prefix + "_process_dev", self._h, _dev_in(x, self.dtype), buffer_size, nb, p("bb"), p("fm"), p("am"),
              p("usb"), int(stride), C.byref(got), _stream_ptr())
    return got.value


ChannelBank.process_into = _bank_process_into


class ShardedChannelBank(ChannelBank):
    """The same bank with its channels sharded by contiguous ranges over the GPUs `devices` of THIS process
    (sdrg_bank_sharded_*): torch tensors in / out live on devices[0]; numpy arrays go through every device's
    own host<->device copies.  Bit-identical to ChannelBank for "s8" / "s16"; for "f32" equal to it to float
    rounding (window sums are float atomics)."""

    _prefix = "sdrg_bank_sharded"

    def __init__(self, scalar, Fc, Ff, width, order, sub_sample, oFs=0.0, devices=(0,)):
        self.scalar = scalar_id(scalar)
        self.dtype = _NP[self.scalar]
        Fc = np.ascontiguousarray(Fc, dtype=np.float64)
        Ff = Fc if Ff is None else np.ascontiguousarray(Ff, dtype=np.float64)
        self.channels = Fc.shape[0]
        self.devices = [int(d) for d in devices]
        self._h = C.c_void_p()
        dp = C.POINTER(C.c_double)
        devs = (C.c_int * len(self.devices))(*self.devices)
        _lib.call("sdrg_bank_sharded_create", self.scalar, self.channels, Fc.ctypes.data_as(dp), Ff.ctypes.data_as(dp),
                  float(width), int(order), int(sub_sample), float(oFs), devs, len(self.devices), C.byref(self._h))

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.load().sdrg_bank_sharded_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def shards(self):
        """[(device, first_channel, n_channels, direct_peer_stores)] per shard."""
        out = []
        n = C.c_size_t(0)
        _lib.call("sdrg_bank_sharded_info", self._h, None, C.byref(n), 0, None, None, None, None)
        for g in range(n.value):
            dev, lo, cnt, direct = C.c_int(0), C.c_size_t(0), C.c_size_t(0), C.c_int(0)
            _lib.call("sdrg_bank_sharded_info", self._h, None, None, g, C.byref(dev), C.byref(lo), C.byref(cnt), C.byref(direct))
            out.append((dev.value, lo.value, cnt.value, bool(direct.value)))
        return out

    def channel_info(self, c):
        raise NotImplementedError("per-channel design lives in the shards; build a ChannelBank to inspect it")


def autocast_cs16(x):
    """AutoCast< complex<int16> > of complex uint8 / int8 samples (n, 2) (src/autocast.hh:187-204)."""
    if _is_torch(x):
        import torch
        t = _lib.T_CU8 if x.dtype == torch.uint8 else _lib.T_CS8
        out = torch.empty(x.shape, dtype=torch.int16, device=x.device)
        _lib.call("sdrg_autocast_process_dev", t, _lib.T_CS16, C.c_void_p(x.data_ptr()), x.shape[0], C.c_void_p(out.data_ptr()), _stream_ptr())
        return out
    x = np.ascontiguousarray(x)
    t = _lib.T_CU8 if x.dtype == np.uint8 else _lib.T_CS8
    out = np.zeros(x.shape, dtype=np.int16)
    _lib.call("sdrg_autocast_process", t, _lib.T_CS16, _np_ptr(x), x.shape[0], _np_ptr(out))
    return out


def autocast(x, in_type, out_type):
    """AutoCast<out_type> (src/autocast.hh:30-69) of a numpy array / CUDA tensor holding elements of `in_type`
    (Config::Type ids, _lib.T_*).  Returns the output as raw uint8 bytes (numpy) or a uint8 tensor."""
    in_elem = [0, 1, 1, 2, 2, 4, 8, 2, 2, 4, 4, 8, 16][int(in_type)]
    nbytes = C.c_size_t(0)
    if _is_torch(x):
        import torch
        raw = x.contiguous().view(torch.uint8).reshape(-1)
        n = raw.numel() // in_elem
        _lib.call("sdrg_autocast_out_bytes", int(in_type), int(out_type), n, C.byref(nbytes))
        out = torch.empty(max(nbytes.value, 1), dtype=torch.uint8, device=x.device)
        _lib.call("sdrg_autocast_process_dev", int(in_type), int(out_type), _dev_in(raw), n, C.c_void_p(out.data_ptr()), _stream_ptr())
        return out[:nbytes.value]
    raw = np.ascontiguousarray(x).view(np.uint8).reshape(-1)
    n = raw.size // in_elem
    _lib.call("sdrg_autocast_out_bytes", int(in_type), int(out_type), n, C.byref(nbytes))
    out = np.zeros(max(nbytes.value, 1), dtype=np.uint8)
    _lib.call("sdrg_autocast_process", int(in_type), int(out_type), _np_ptr(raw), n, _np_ptr(out))
    return out[:nbytes.value]


class FMDeemph:
    """FMDeemph<int16_t> (src/demod.hh:271-362) for `streams` independent audio streams (rows)."""

    def __init__(self, streams=1):
        self.streams = int(streams)
        self._h = C.c_void_p()
        _lib.call("sdrg_fmdeemph_create", self.streams, C.byref(self._h))

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.load().sdrg_fmdeemph_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def config(self, src_cfg=None, *, sample_rate=0.0, buffer_size=0, type=_lib.T_S16):
        if src_cfg is None:
            src_cfg = Config(type, sample_rate, buffer_size, 1)
        out = Config()
        _lib.call("sdrg_fmdeemph_configure", self._h, C.byref(src_cfg), C.byref(out))
        return out

    def process(self, x):
        """x: (streams, n) int16 (or (n,) for one stream)."""
        if _is_torch(x):
            import torch
            x2 = x.view(self.streams, -1)
            out = torch.empty_like(x2)
            _lib.call("sdrg_fmdeemph_process_dev", self._h, C.c_void_p(x2.data_ptr()), x2.shape[1], x2.stride(0),
                      C.c_void_p(out.data_ptr()), _stream_ptr())
            return out.view(x.shape)
        x2 = np.ascontiguousarray(x, dtype=np.int16).reshape(self.streams, -1)
        out = np.zeros_like(x2)
        _lib.call("sdrg_fmdeemph_process", self._h, _np_ptr(x2), x2.shape[1], x2.shape[1], _np_ptr(out))
        return out.reshape(np.shape(x))
