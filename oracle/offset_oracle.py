"""CPU oracle of the channel-alignment functions (reference passiveRadar/signal_utils.py:29-78).

* ``*_oracle``: the reference's arithmetic restated with the same SciPy calls (scipy.signal.decimate,
  np.pad, scipy.signal.correlate, np.argmax), so the outputs equal the reference's bit for bit.
* ``*_truth``: the same quantities in float64 throughout -- float64 filter coefficients and filtering,
  float64 FFT correlation -- to tell the device's round-off from the reference's own.

Test infrastructure only; the product package never imports it.
"""
from __future__ import annotations

import numpy as np
import scipy.signal as signal


def xcorr_oracle(s1, s2, nlead, nlag):
    return signal.correlate(s1, np.pad(s2, (nlag, nlead), mode='constant'), mode='valid')


def channel_offset_oracle(s1, s2, nd, nl):
    """(offset, |xc|) exactly as find_channel_offset computes them."""
    B1 = signal.decimate(s1, nd)
    B2 = np.pad(signal.decimate(s2, nd), (nl, nl), 'constant')
    xc = np.abs(signal.correlate(B1, B2, mode='valid'))
    return (np.argmax(xc) - nl) * nd, xc


def offset_compensation_oracle(x1, x2, ns, ndec, nlag=2000):
    os_, _ = channel_offset_oracle(x1[0:int(ns)], x2[0:int(ns)], ndec, nlag)
    if os_ == 0:
        return x2
    e = np.zeros_like(x2)
    if os_ > 0:
        e[os_:] = x2[:-os_]
    else:
        e[:os_] = x2[-os_:]
    return e


PADLEN = 27          # sosfiltfilt's odd extension for decimate's 4 sections


def decimate_truth(x, nd):
    """decimate's zero-phase IIR filter in float64 (complex128 for complex inputs).  Integer inputs keep the
    reference's odd extension, which decimate computes in the integer dtype (it wraps around); only the filter
    runs in float64."""
    x = np.asarray(x)
    sos = signal.cheby1(8, 0.05, 0.8 / nd, output='sos')
    if np.issubdtype(x.dtype, np.integer):
        P = PADLEN
        ext = np.concatenate([2 * x[:1] - x[P:0:-1], x, 2 * x[-1:] - x[-2:-P - 2:-1]])
        return signal.sosfiltfilt(sos, ext.astype(np.float64), padlen=0)[P:-P][::nd]
    x = x.astype(np.complex128 if np.iscomplexobj(x) else np.float64)
    return signal.sosfiltfilt(sos, x)[::nd]


def corr_truth(x, y, lag0, nlags):
    """out[k] = sum_i x[i] conj(y[i + lag0 - k]), k < nlags, by a float64 FFT."""
    x = np.asarray(x, dtype=np.complex128)
    y = np.asarray(y, dtype=np.complex128)
    full = signal.fftconvolve(x, np.conj(y[::-1]), mode='full')     # full[j] = c[(len(y) - 1) - j]
    lags = lag0 - np.arange(nlags)
    j = (y.shape[0] - 1) - lags
    out = np.zeros(nlags, dtype=np.complex128)
    ok = (j >= 0) & (j < full.shape[0])
    out[ok] = full[j[ok]]
    return out


def xcorr_truth(s1, s2, nlead, nlag):
    n1, n2 = len(s1), len(s2)
    L2 = n2 + nlag + nlead
    lag0, nlags = (n2 - n1 + nlead, L2 - n1 + 1) if L2 >= n1 else (-nlag, n1 - L2 + 1)
    return corr_truth(s1, s2, lag0, nlags)


def channel_offset_truth(s1, s2, nd, nl):
    """(offset, |xc|, B1, B2) with float64 filtering and a float64 correlation; |Re xc| for real inputs."""
    B1, B2 = decimate_truth(s1, nd), decimate_truth(s2, nd)
    c = xcorr_truth(B1, B2, nl, nl)
    xc = np.abs(c) if np.iscomplexobj(B1) or np.iscomplexobj(B2) else np.abs(c.real)
    return (int(np.argmax(xc)) - nl) * nd, xc, B1, B2
