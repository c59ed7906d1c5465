"""Seeded synthetic two-channel IQ used by the tests, the goldens and bench.py.

The reference ships no recordings (its README points at a 6 GB Google-Drive
file), so every measurement in this repo runs on synthetic complex64 IQ with
the shapes BASELINE.json names.  Two profiles (SURVEY.md section 8d):

* ``P0``  reference and surveillance channels are independent unit-power white
  noise.  Strict-parity profile: nothing cancels, so float32 round-off of the
  reference implementation itself stays at the 1e-7 level.
* ``P1``  surveillance = direct-path + multipath clutter (delayed, scaled copies
  of the illuminator) + one weak Doppler-shifted target + receiver noise.  This
  is what a passive radar actually sees and what the LS / NLMS cancellers are
  for.

Pure host-side numpy; nothing here is on the timed path.
"""
from __future__ import annotations

import numpy as np

BASE_SEED = 20260924

# (delay in samples, complex amplitude) of the static clutter taps of profile P1
P1_CLUTTER = ((0, 1.0 + 0.0j), (3, 0.5j), (17, -0.2 + 0.0j), (60, 0.05 + 0.05j))
P1_TARGET = dict(delay=40, doppler_hz=37.0, amplitude=1e-3)
P1_NOISE_SIGMA = 1e-3
P1_SAMPLE_RATE = float(2 ** 19)


def white_iq(rng: np.random.Generator, n: int) -> np.ndarray:
    """Unit-power circular white noise, complex64."""
    re = rng.standard_normal(n, dtype=np.float32)
    im = rng.standard_normal(n, dtype=np.float32)
    out = np.empty(n, dtype=np.complex64)
    out.real = re
    out.imag = im
    out *= np.float32(1.0 / np.sqrt(2.0))
    return out


def make_frame(n: int, profile: str = "P1", frame: int = 0, seed: int = BASE_SEED):
    """Return ``(ref, srv)`` complex64 arrays of length ``n`` for CPI frame ``frame``."""
    rng = np.random.default_rng(seed + frame)
    ref = white_iq(rng, n)
    if profile == "P0":
        srv = white_iq(rng, n)
        return ref, srv
    if profile != "P1":
        raise ValueError(f"unknown profile {profile!r}")
    noise = white_iq(rng, n)
    acc = np.zeros(n, dtype=np.complex128)
    for delay, amp in P1_CLUTTER:
        acc += amp * np.roll(ref, delay % n if n else 0)
    t = P1_TARGET
    phase = 2.0 * np.pi * t["doppler_hz"] * np.arange(n, dtype=np.float64) / P1_SAMPLE_RATE
    acc += t["amplitude"] * np.roll(ref, t["delay"] % n if n else 0) * np.exp(1j * phase)
    acc += P1_NOISE_SIGMA * noise
    return ref, acc.astype(np.complex64)


def frame_digest(ref: np.ndarray, srv: np.ndarray) -> np.ndarray:
    """Small fingerprint stored next to goldens to detect RNG-stream drift."""
    n = ref.shape[0]
    picks = np.unique(np.clip(np.array([0, 1, n // 3, n // 2, n - 1]), 0, max(n - 1, 0)))
    return np.concatenate([
        ref[picks], srv[picks],
        np.array([ref.astype(np.complex128).sum(), srv.astype(np.complex128).sum()]).astype(np.complex64),
    ])


def raw_iq(n, kind="int8", seed=11):
    """Seeded interleaved I/Q block of ``n`` complex samples as a receiver would deliver it
    (``int8``: HackRF-style, ``int16``, or ``float32``); input of the front-end chain."""
    rng = np.random.default_rng(seed)
    if kind == "int8":
        return rng.integers(-128, 128, size=2 * n, dtype=np.int8)
    if kind == "int16":
        return rng.integers(-2048, 2048, size=2 * n, dtype=np.int16)
    if kind == "float32":
        return rng.standard_normal(2 * n).astype(np.float32)
    raise ValueError(f"unknown raw IQ kind {kind!r}")


def offset_pair(n, offset, kind="complex64", seed=BASE_SEED + 73, snr_db=10.0):
    """Two receiver channels of one band-limited FM-like broadcast, ``offset`` samples apart, each with its own
    noise: ``s1[i] = s[i] + e1[i]`` and ``s2[i] = s[i + offset] + e2[i]``, so ``find_channel_offset(s1, s2, ...)``
    finds ``offset``.  The smooth instantaneous frequency keeps the band narrow, so the correlation peak is broad
    as on recorded data.  ``kind``: ``complex64`` (complex baseband), or ``int8`` / ``int16`` (a real band-pass
    signal quantised as a receiver delivers raw samples)."""
    rng = np.random.default_rng(seed)
    total = n + abs(int(offset))
    knots = rng.standard_normal(total // 64 + 2)
    msg = np.interp(np.arange(total) / 64.0, np.arange(knots.size), knots)
    real = kind in ("int8", "int16")
    freq = (0.12 if real else 0.0) + 0.06 * msg                  # cycles per sample
    phase = 2.0 * np.pi * np.cumsum(freq)
    s = np.cos(phase) if real else np.exp(1j * phase)
    a = max(0, -int(offset))
    sigma = 10.0 ** (-snr_db / 20.0)

    def noise():
        if real:
            return sigma * rng.standard_normal(n)
        return sigma * (rng.standard_normal(n) + 1j * rng.standard_normal(n)) / np.sqrt(2.0)

    s1 = s[a:a + n] + noise()
    s2 = s[a + offset:a + offset + n] + noise()
    if kind == "complex64":
        return s1.astype(np.complex64), s2.astype(np.complex64)
    if real:
        scale, lim, dt = (40.0, 127, np.int8) if kind == "int8" else (4000.0, 32767, np.int16)
        q = lambda v: np.clip(np.round(v * scale), -lim - 1, lim).astype(dt)
        return q(s1), q(s2)
    raise ValueError(f"unknown kind {kind!r}")
