"""Front-end signal utilities on the B200 -- same call signatures as the reference.

Drop-ins for ``passiveRadar.signal_utils.deinterleave_IQ`` (reference
``passiveRadar/signal_utils.py:19-22``), ``frequency_shift`` (``:24-27``) and ``resample``
(``:15-17``), the chain ``main.py:105-166`` runs on every input chunk, plus ``frontend`` which runs
the three in one pass on the device (raw IQ in, resampled complex64 out).  All arithmetic runs in
``libprcore.so``; no CPU fallback.

Also the channel alignment main.py runs once per run (main.py:54, :83): ``find_channel_offset`` (``:73-78``),
``offset_compensation`` (``:49-71``) and the long-lag correlation ``xcorr`` (``:29-32``) they rest on.
"""
from __future__ import annotations

import functools
import math
import operator

import numpy as np

from . import _lib


def _is_weak(v):
    """Does ``v`` stay 'weak' in the reference's expression (NumPy 2 promotion)?  Python scalars do;
    so does ``np.float64`` there, because it subclasses ``float`` and ``1j*2*np.pi*fc`` /
    ``1j*phase_offset`` are evaluated by Python's ``complex.__mul__`` before NumPy sees them.
    Arrays (what main.py passes as phase_offset) and other NumPy scalar types are strong."""
    return isinstance(v, (bool, int, float, np.float32))


def _is_weak_divisor(v):
    """``array / Fs``: here NumPy does see the scalar, and a NumPy float64 scalar is strong."""
    return isinstance(v, (bool, int, float)) and not isinstance(v, np.generic)


def _raw_iq(interleavedIQ):
    """interleaved real array -> (buffer, in_kind, n complex samples); I = x[0:-1:2], Q = x[1::2]."""
    x = np.asarray(interleavedIQ)
    if x.ndim != 1:
        raise ValueError("interleaved IQ must be one-dimensional")
    n = x.shape[0] // 2
    x = x[:2 * n]
    if x.dtype == np.int8:
        return np.ascontiguousarray(x), _lib.IQ_I8, n
    if x.dtype == np.int16:
        return np.ascontiguousarray(x), _lib.IQ_I16, n
    return np.ascontiguousarray(x, dtype=np.float32), _lib.IQ_C64, n


def _mix_mode(fc, Fs, phase_offset):
    po = np.asarray(phase_offset)
    if po.size != 1:
        raise ValueError("phase_offset must be a scalar (or a one-element array, as main.py passes)")
    if np.iscomplexobj(po):
        raise TypeError("phase_offset must be real")
    if not _is_weak(fc):
        return _lib.MIX_F64, float(po.reshape(()))
    if not _is_weak_divisor(Fs):
        return _lib.MIX_FS64, float(po.reshape(()))
    if _is_weak(phase_offset):
        return _lib.MIX_C64, float(phase_offset)
    return _lib.MIX_C128, float(po.reshape(()))


def deinterleave_IQ(interleavedIQ, *, device=None):
    '''convert interleaved IQ samples to complex64'''
    buf, kind, n = _raw_iq(interleavedIQ)
    out = np.empty(n, dtype=np.complex64)
    if n == 0:
        return out
    lib = _lib.load()
    dev = _lib.current_device() if device is None else int(device)
    _lib.check(lib.prc_iq_mix_c64(buf.ctypes.data, kind, n, _lib.MIX_NONE, 0.0, 1.0, 0.0, out.ctypes.data,
                                  _lib.MEM_HOST, dev, None, 0))
    return out


def frequency_shift(x, fc, Fs, phase_offset=0, *, device=None):
    '''frequency shift x by fc where Fs is the sample rate of x

    The reference builds the phase ramp from ``arange(..., dtype=complex64)``, i.e. in float32; the
    device kernel reproduces that rounding (it is what the reference's output actually contains).
    Returns complex64 when the reference would (complex64 ``x``, Python-scalar arguments), else
    complex128 (the device result widened).'''
    x = np.asarray(x)
    if x.ndim != 1:
        raise ValueError("x must be one-dimensional")
    mode, po = _mix_mode(fc, Fs, phase_offset)
    xin = _lib.as_c64(x, "x")
    n = xin.shape[0]
    out = np.empty(n, dtype=np.complex64)
    if n:
        lib = _lib.load()
        dev = _lib.current_device() if device is None else int(device)
        _lib.check(lib.prc_iq_mix_c64(xin.ctypes.data, _lib.IQ_C64, n, mode, float(fc), float(Fs), po,
                                      out.ctypes.data, _lib.MEM_HOST, dev, None, 0))
    narrow = mode == _lib.MIX_C64 and x.dtype in (np.complex64, np.float32, np.float16)
    return out if narrow else out.astype(np.complex128)


@functools.lru_cache(maxsize=32)
def _resample_taps(up, dn, single):
    """The low-pass resample_poly designs (scipy/signal/_signaltools.py, resample_poly), times ``up``;
    float32-rounded first when the signal is complex64 (``h = asarray(h, dtype=x.dtype)``)."""
    from scipy.signal import firwin
    max_rate = max(up, dn)
    half_len = 10 * max_rate
    h = firwin(2 * half_len + 1, 1.0 / max_rate, window=('kaiser', 5.0))
    if single:
        h = (h.astype(np.float32) * np.float32(up)).astype(np.float64)
    else:
        h = h * up
    return np.ascontiguousarray(h, dtype=np.float64)


def _reduced(up, dn):
    if up != int(up):
        raise ValueError("up must be an integer")
    if dn != int(dn):
        raise ValueError("down must be an integer")
    up, dn = int(up), int(dn)
    if up < 1 or dn < 1:
        raise ValueError('up and down must be >= 1')
    g = math.gcd(up, dn)
    return up // g, dn // g


def _run_frontend(buf, kind, n, mode, fc, Fs, po, up, dn, single, device):
    h = _resample_taps(up, dn, single)
    n_out = n * up
    n_out = n_out // dn + bool(n_out % dn)
    out = np.empty(n_out, dtype=np.complex64)
    lib = _lib.load()
    dev = _lib.current_device() if device is None else int(device)
    _lib.check(lib.prc_frontend_c64(buf.ctypes.data, kind, n, mode, float(fc), float(Fs), po, up, dn,
                                    h.ctypes.data, h.shape[0], out.ctypes.data, n_out, _lib.MEM_HOST, dev, None, 0))
    return out


def resample(x, up, dn, *, device=None):
    '''rational resampling by a factor of up/dn  (scipy.signal.resample_poly(x, up, dn, padtype='line'))'''
    x = np.asarray(x)
    if x.ndim != 1:
        raise ValueError("x must be one-dimensional")
    up, dn = _reduced(up, dn)
    if up == dn == 1:
        return x.copy()
    if x.shape[0] == 0:
        raise ValueError("x must not be empty")
    single = x.dtype in (np.complex64, np.float32)
    out = _run_frontend(_lib.as_c64(x, "x"), _lib.IQ_C64, x.shape[0], _lib.MIX_NONE, 0.0, 1.0, 0.0, up, dn, single, device)
    if np.iscomplexobj(x):
        return out if x.dtype == np.complex64 else out.astype(np.complex128)
    return out.real.astype(x.dtype if x.dtype.kind == 'f' else np.float64)


def frontend(interleavedIQ, fc, Fs, phase_offset, up, dn, *, device=None):
    '''``resample(frequency_shift(deinterleave_IQ(interleavedIQ), fc, Fs, phase_offset), up, dn)`` in one
    pass on the device: the raw samples cross PCIe once (2 bytes per sample for int8 IQ) and only the
    resampled complex64 block comes back.  Not a reference function; it is the composition
    ``main.py:105-166`` applies to every chunk.'''
    buf, kind, n = _raw_iq(interleavedIQ)
    if n == 0:
        raise ValueError("interleavedIQ must hold at least one I/Q pair")
    mode, po = _mix_mode(fc, Fs, phase_offset)
    up, dn = _reduced(up, dn)
    if up == dn == 1:
        out = np.empty(n, dtype=np.complex64)
        lib = _lib.load()
        dev = _lib.current_device() if device is None else int(device)
        _lib.check(lib.prc_iq_mix_c64(buf.ctypes.data, kind, n, mode, float(fc), float(Fs), po, out.ctypes.data,
                                      _lib.MEM_HOST, dev, None, 0))
        return out
    # the reference chain is complex64 end to end only with Python-scalar arguments
    return _run_frontend(buf, kind, n, mode, fc, Fs, po, up, dn, mode == _lib.MIX_C64, device)


# ---------------------------------------------------------------------------------------------------- long-lag xcorr
def _xcorr_window(n1, n2, nlead, nlag):
    """(lag0, nlags) of ``correlate(s1, pad(s2, (nlag, nlead)), 'valid')``: out[k] = c[lag0 - k] with
    c[m] = sum_i s1[i] conj(s2[i + m]) (include/prcore.h, prc_xcorr_c64)."""
    L2 = n2 + nlag + nlead
    if L2 >= n1:
        return n2 - n1 + nlead, L2 - n1 + 1
    return -nlag, n1 - L2 + 1


def _pad_width(v):
    """np.pad's checks of one pad width: integral (TypeError), non-negative (ValueError)."""
    try:
        v = operator.index(v)
    except TypeError:
        raise TypeError("`pad_width` must be of integral type.") from None
    if v < 0:
        raise ValueError("index can't contain negative values")
    return v


_XCORR_DTYPES = (np.float32, np.float64, np.complex64, np.complex128)


def xcorr(s1, s2, nlead, nlag, *, device=None):
    ''' cross-correlate s1 and s2 with sample offsets from -1*nlag to nlead

    ``scipy.signal.correlate(s1, np.pad(s2, (nlag, nlead)), 'valid')`` as one lag window of a circular FP32
    transform on the device.  The result dtype is SciPy's (float32 / float64 / complex64 / complex128); 64-bit
    results are the complex64 device result widened.  Integer inputs raise TypeError: SciPy's direct integer path
    can overflow, and no caller in the reference passes integers.'''
    s1 = np.asarray(s1)
    s2 = np.asarray(s2)
    for name, a in (("s1", s1), ("s2", s2)):
        if a.ndim != 1:
            raise ValueError(f"{name} must be one-dimensional")
        if a.dtype.type not in _XCORR_DTYPES:
            raise TypeError(f"{name}: dtype {a.dtype} not supported (float32, float64, complex64, complex128)")
        if a.shape[0] == 0:
            raise ValueError(f"{name} must not be empty")
    nlead, nlag = _pad_width(nlead), _pad_width(nlag)
    lag0, nlags = _xcorr_window(s1.shape[0], s2.shape[0], nlead, nlag)
    x = np.ascontiguousarray(s1, dtype=np.complex64)
    y = np.ascontiguousarray(s2, dtype=np.complex64)
    out = np.empty(nlags, dtype=np.complex64)
    lib = _lib.load()
    dev = _lib.current_device() if device is None else int(device)
    _lib.check(lib.prc_xcorr_c64(x.ctypes.data, x.shape[0], y.ctypes.data, y.shape[0], lag0, nlags, out.ctypes.data,
                                 _lib.MEM_HOST, dev, None, 0))
    rt = np.result_type(s1.dtype, s2.dtype)
    if rt.kind == 'c':
        return out if rt == np.complex64 else out.astype(rt)
    return out.real.astype(rt)


def _decimate_type(dtype):
    """scipy.signal.decimate's working dtype: integers (and float16) are upcast to float64."""
    if not np.issubdtype(dtype, np.inexact) or dtype == np.float16:
        return np.dtype(np.float64)
    return np.dtype(dtype)


@functools.lru_cache(maxsize=32)
def _decimate_sos(q, single):
    """The IIR sections scipy.signal.decimate(x, q) designs (cheby1(8, 0.05, 0.8 / q, output='sos')), rounded to
    float32 when decimate casts them to a float32 / complex64 signal's dtype; and sosfiltfilt's padlen."""
    from scipy.signal import cheby1
    sos = cheby1(8, 0.05, 0.8 / q, output='sos')
    if single:
        sos = sos.astype(np.float32).astype(np.float64)
    ntaps = 2 * sos.shape[0] + 1 - min(int((sos[:, 2] == 0).sum()), int((sos[:, 5] == 0).sum()))
    return np.ascontiguousarray(sos, dtype=np.float64), 3 * ntaps


def _offset_operands(s1, s2):
    """Both channels in one device input kind (PRC_SIG_*) and the dtype decimate would work in."""
    s1 = np.asarray(s1)
    s2 = np.asarray(s2)
    for name, a in (("s1", s1), ("s2", s2)):
        if a.ndim != 1:
            raise ValueError(f"{name} must be one-dimensional")
    if s1.dtype == s2.dtype and s1.dtype in (np.int8, np.int16):
        kind = _lib.SIG_I8 if s1.dtype == np.int8 else _lib.SIG_I16
        return np.ascontiguousarray(s1), np.ascontiguousarray(s2), kind, np.dtype(np.float64)
    wt = np.result_type(_decimate_type(s1.dtype), _decimate_type(s2.dtype))
    if wt.kind == 'c':
        dt, kind = (np.complex64, _lib.SIG_C64) if wt == np.complex64 else (np.complex128, _lib.SIG_C128)
    else:
        dt, kind = np.float64, _lib.SIG_F64
    return np.ascontiguousarray(s1, dtype=dt), np.ascontiguousarray(s2, dtype=dt), kind, wt


def find_channel_offset(s1, s2, nd, nl, *, device=None, return_xc=False):
    '''use cross-correlation to find channel offset in samples

    ``(argmax |correlate(decimate(s1, nd), pad(decimate(s2, nd), (nl, nl)), 'valid')| - nl) * nd`` with
    decimate's zero-phase Chebyshev-I filter run in float64 on the device and the 2 nl + 1 lags correlated there
    as well; only the offset comes back.  The reference's argument errors are raised before the device is used.
    ``return_xc=True`` also returns the float32 |xc| vector.'''
    q = operator.index(nd)
    s1, s2, kind, wt = _offset_operands(s1, s2)
    sos, padlen = _decimate_sos(q, wt in (np.float32, np.complex64))
    for a in (s1, s2):
        if a.shape[0] <= padlen:
            raise ValueError("The length of the input vector x must be greater than padlen, which is %d." % padlen)
    nl = _pad_width(nl)
    n1d, n2d = -(-s1.shape[0] // q), -(-s2.shape[0] // q)
    _, nlags = _xcorr_window(n1d, n2d, nl, nl)
    off = np.zeros(1, dtype=np.int64)
    xc = np.empty(nlags, dtype=np.float32) if return_xc else None
    lib = _lib.load()
    dev = _lib.current_device() if device is None else int(device)
    _lib.check(lib.prc_channel_offset(s1.ctypes.data, s1.shape[0], s2.ctypes.data, s2.shape[0], kind, q, nl,
                                      sos.ctypes.data, sos.shape[0], off.ctypes.data, _lib.ptr(xc),
                                      _lib.MEM_HOST, dev, None, 0))
    return (off[0], xc) if return_xc else off[0]


def _shift(x, n):
    """x delayed by n samples (advanced for n < 0), zero filled, same dtype."""
    e = np.zeros_like(x)
    m = x.shape[0]
    if n > 0 and n < m:
        e[n:] = x[:m - n]
    elif n < 0 and -n < m:
        e[:m + n] = x[-n:]
    return e


def offset_compensation(x1, x2, ns, ndec, nlag=2000, *, device=None):
    '''Find and correct a constant time offset between two signals using a
    cross-correlation

    The offset comes from the device (find_channel_offset on the first ``int(ns)`` samples); the zero-filled
    shift of x2 is a host copy.  An offset of 0 returns x2 itself, as the reference does.'''
    s1 = x1[0:int(ns)]
    s2 = x2[0:int(ns)]
    os_ = find_channel_offset(s1, s2, ndec, nlag, device=device)
    if os_ == 0:
        return x2
    return _shift(np.asarray(x2), int(os_))
