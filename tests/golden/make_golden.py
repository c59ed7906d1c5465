#!/usr/bin/env python
"""Generate the golden vectors under tests/golden/ by EXECUTING THE REFERENCE.

Run in the build container (where /root/reference exists):

    python tests/golden/make_golden.py [--big]

Every array written here is an output of the reference's own functions
(``passiveRadar.range_doppler_processing.fast_xambg``,
``passiveRadar.clutter_removal.{LS_Filter, NLMS_filter}``) imported from
``/root/reference`` -- nothing from ``oracle/`` or ``passiveradar_b200/csrc`` is
involved, only the seeded input generator ``passiveradar_b200.synth``.

Cases tagged ``literal`` call the reference untouched.  Cases tagged ``shim``
call the same reference function while ``scipy.signal.decimate`` is patched so
that an FIR ``dlti`` goes straight to ``resample_poly`` (what SciPy does anyway,
scipy/signal/_signaltools.py:5344-5347) instead of first running
``dlti._as_zpk()`` -> ``np.roots`` of degree ``ndecim`` once per range lag
(16 s/lag at ndecim=3125, 46 s/lag at 4096).  The case ``xambg_shim_proof``
stores both outputs for one input so the tests can assert they are identical.

The GPU box has no /root/reference; it only ever reads the .npz files.
"""
from __future__ import annotations

import argparse
import contextlib
import os
import sys
import time

# before numpy loads OpenBLAS: the goldens' BLAS configuration (tests/_golden.py GOLDEN_BLAS)
os.environ.update(OPENBLAS_CORETYPE="SkylakeX", OPENBLAS_NUM_THREADS="8")

import numpy as np  # noqa: E402
import scipy.signal as signal

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.environ.get("PR_REFERENCE", "/root/reference"))

from passiveRadar.range_doppler_processing import fast_xambg          # noqa: E402  (the reference)
from passiveRadar.clutter_removal import LS_Filter, NLMS_filter, LS_Filter_Toeplitz, LS_Filter_Multiple   # noqa: E402  (the reference)
from passiveRadar.signal_utils import frequency_shift, deinterleave_IQ, resample   # noqa: E402  (the reference)
from passiveRadar.range_doppler_processing import direct_xambg        # noqa: E402  (the reference)
from passiveradar_b200 import synth                                    # noqa: E402


@contextlib.contextmanager
def fir_decimate_shim():
    real = signal.decimate

    def patched(x, q, n=None, ftype='iir', axis=-1, zero_phase=True):
        if isinstance(ftype, signal.dlti) and zero_phase:
            tf = ftype._as_tf()
            den = np.atleast_1d(tf.den)
            if den.shape[0] == 1:                      # FIR
                return signal.resample_poly(x, 1, q, axis=axis, window=tf.num / tf.den)
        return real(x, q, n=n, ftype=ftype, axis=axis, zero_phase=zero_phase)

    signal.decimate = patched
    try:
        yield
    finally:
        signal.decimate = real


OUT_DIR = os.environ.get("PR_GOLDEN_OUT", HERE)       # tests regenerate into a scratch directory


def save(name, **arrays):
    path = os.path.join(OUT_DIR, name + ".npz")
    np.savez_compressed(path, **arrays)
    print(f"  wrote {name}.npz ({os.path.getsize(path) / 1024:.1f} KiB)")


def kaiser(n):
    return signal.get_window(('kaiser', 5.0), n)


def xambg_case(name, n, F, R, profile, window, literal, input_len=None, short_filt=True,
               n_given=None, store_inputs=True, frame=0):
    n_given = n if n_given is None else n_given
    ref, srv = synth.make_frame(n_given, profile, frame)
    if window == 'kaiser':
        win_arg = kaiser(n)
    elif window == 'tuple':
        win_arg = ('kaiser', 5.0)
    else:
        win_arg = None
    t0 = time.time()
    if literal:
        out = fast_xambg(ref, srv, R, F, input_len, win_arg, short_filt)
    else:
        with fir_decimate_shim():
            out = fast_xambg(ref, srv, R, F, input_len, win_arg, short_filt)
    dt = time.time() - t0
    arrays = dict(n=n_given, F=F, R=R, profile=profile, window='none' if window is None else window, literal=literal,
                  input_len=-1 if input_len is None else input_len, short_filt=short_filt,
                  frame=frame, out=out, digest=synth.frame_digest(ref, srv), seconds=dt)
    if store_inputs:
        arrays.update(ref=ref, srv=srv)
    print(f"{name}: n={n_given} F={F} R={R} {profile} window={window} literal={literal} {dt:.2f}s")
    save(name, **arrays)


def subsample_idx(n, count=4096):
    step = max(1, n // count)
    return np.arange(0, n, step)


def ls_case(name, n, filter_len, reg, peek, profile, store_inputs=True, frame=0):
    ref, srv = synth.make_frame(n, profile, frame)
    t0 = time.time()
    out, taps = LS_Filter(ref, srv, filter_len, reg, peek, True)
    dt = time.time() - t0
    idx = subsample_idx(n)
    arrays = dict(n=n, filter_len=filter_len, reg=reg, peek=peek, profile=profile, frame=frame,
                  taps=taps, digest=synth.frame_digest(ref, srv), seconds=dt,
                  out_idx=idx, out_sub=out[idx],
                  out_sum=np.complex128(out.astype(np.complex128).sum()),
                  out_abs2=np.float64((np.abs(out.astype(np.complex128)) ** 2).sum()),
                  srv_absmax=np.float64(np.abs(srv).max()))
    if store_inputs:
        arrays.update(ref=ref, srv=srv, out=out)
    print(f"{name}: n={n} filterLen={filter_len} reg={reg} peek={peek} {profile} {dt:.2f}s")
    save(name, **arrays)


def toeplitz_case(name, n, filter_len, peek, profile, store_inputs=True, frame=0):
    ref, srv = synth.make_frame(n, profile, frame)
    t0 = time.time()
    out, taps = LS_Filter_Toeplitz(ref, srv, filter_len, peek, True)
    dt = time.time() - t0
    idx = subsample_idx(n)
    arrays = dict(n=n, filter_len=filter_len, peek=peek, profile=profile, frame=frame, taps=taps,
                  digest=synth.frame_digest(ref, srv), seconds=dt, out_idx=idx, out_sub=out[idx],
                  out_sum=np.complex128(out.sum()), srv_absmax=np.float64(np.abs(srv).max()))
    if store_inputs:
        arrays.update(ref=ref, srv=srv, out=out)
    print(f"{name}: n={n} filterLen={filter_len} peek={peek} {profile} {dt:.2f}s")
    save(name, **arrays)


def multiple_case(name, n, filter_len, sample_rate, bins, profile, store_inputs=True, frame=0):
    ref, srv = synth.make_frame(n, profile, frame)
    t0 = time.time()
    out = LS_Filter_Multiple(ref, srv, filter_len, sample_rate, list(bins))
    dt = time.time() - t0
    idx = subsample_idx(n)
    arrays = dict(n=n, filter_len=filter_len, sample_rate=sample_rate, bins=np.array(bins, dtype=np.float64),
                  profile=profile, frame=frame, digest=synth.frame_digest(ref, srv), seconds=dt,
                  out_idx=idx, out_sub=out[idx], out_sum=np.complex128(out.sum()),
                  srv_absmax=np.float64(np.abs(srv).max()),
                  shift_sample=frequency_shift(ref, bins[-1], sample_rate)[idx])
    if store_inputs:
        arrays.update(ref=ref, srv=srv, out=out)
    print(f"{name}: n={n} filterLen={filter_len} Fs={sample_rate} bins={list(bins)} {profile} {dt:.2f}s")
    save(name, **arrays)


def nlms_case(name, n, filter_len, mu, peek, profile, with_init=False, frame=0):
    ref, srv = synth.make_frame(n, profile, frame)
    init = None
    if with_init:
        rng = np.random.default_rng(77)
        init = (0.01 * (rng.standard_normal(filter_len + peek)
                        + 1j * rng.standard_normal(filter_len + peek))).astype(np.complex64)
    t0 = time.time()
    out, w = NLMS_filter(ref, srv, filter_len, mu, peek, init, True)
    dt = time.time() - t0
    arrays = dict(n=n, filter_len=filter_len, mu=mu, peek=peek, profile=profile, frame=frame,
                  ref=ref, srv=srv, out=out, taps=w, seconds=dt,
                  init=np.zeros(0, np.complex64) if init is None else init)
    print(f"{name}: n={n} filterLen={filter_len} mu={mu} peek={peek} init={with_init} {dt:.2f}s")
    save(name, **arrays)


def frame_case(name, n, F, R, profile, store_inputs, frame=0):
    """Chained LS_Filter -> fast_xambg (filterLen = R as main.py:172 does)."""
    ref, srv = synth.make_frame(n, profile, frame)
    t0 = time.time()
    cleaned, taps = LS_Filter(ref, srv, R, 1.0, 10, True)
    with fir_decimate_shim():
        out = fast_xambg(ref, cleaned, R, F, n, kaiser(n))
    dt = time.time() - t0
    arrays = dict(n=n, F=F, R=R, profile=profile, frame=frame, taps=taps, out=out,
                  digest=synth.frame_digest(ref, srv), seconds=dt)
    if store_inputs:
        arrays.update(ref=ref, srv=srv)
    print(f"{name}: n={n} F={F} R={R} {profile} {dt:.2f}s")
    save(name, **arrays)


def load_reference_cfar():
    """passiveRadar/target_detection.py uses np.float / np.int (removed in NumPy 1.24) in module-level dtype
    tables that CFAR_2D never touches; alias it for the import only -- CFAR_2D itself runs unmodified."""
    import builtins
    added = []
    for alias in ("float", "int", "bool", "complex", "object"):
        if alias not in np.__dict__:
            setattr(np, alias, getattr(builtins, alias))
            added.append(alias)
    try:
        from passiveRadar.target_detection import CFAR_2D
    finally:
        for alias in added:
            delattr(np, alias)
    return CFAR_2D


def cfar_map(rows, cols, seed):
    rng = np.random.default_rng(seed)
    x = np.abs(rng.standard_normal((rows, cols)) + 1j * rng.standard_normal((rows, cols))).astype(np.float32)
    for (r, c, a) in [(rows // 2, cols // 3, 40.0), (3, cols - 2, 25.0), (rows - 1, 0, 30.0)]:
        x[r % rows, c % cols] += np.float32(a)
    return x


def cfar_case(name, rows, cols, fw, gw, thresh=None, seed=5):
    CFAR_2D = load_reference_cfar()
    x = cfar_map(rows, cols, seed)
    out = CFAR_2D(x, fw, gw, thresh)
    print(f"{name}: {rows}x{cols} fw={fw} gw={gw} thresh={thresh} -> {out.dtype}")
    save(name, x=x, fw=fw, gw=gw, thresh=np.float64(-1.0 if thresh is None else thresh), has_thresh=thresh is not None,
         out=out)


def direct_case(name, n, R, F, fs, profile, frame=0):
    ref, srv = synth.make_frame(n, profile, frame)
    t0 = time.time()
    out = direct_xambg(ref, srv, R, F, fs)
    print(f"{name}: n={n} R={R} F={F} fs={fs} {profile} {time.time() - t0:.2f}s")
    save(name, n=n, R=R, F=F, fs=np.float64(fs), profile=profile, frame=frame, digest=synth.frame_digest(ref, srv), out=out)


raw_iq = synth.raw_iq


def front_case(name, n, kind, fc, fs, phase_offset, up, dn, seed=11, store_full=True, po_array=True):
    iq = raw_iq(n, kind, seed)
    po = np.array([phase_offset]) if po_array else phase_offset       # main.py:127-130 passes a (1,) float64 block
    t0 = time.time()
    x = deinterleave_IQ(iq)
    xs = frequency_shift(x, fc, fs, po)
    y = resample(xs, up, dn)
    dt = time.time() - t0
    idx = subsample_idx(n)
    oidx = subsample_idx(y.shape[0])
    arrays = dict(n=n, kind=kind, fc=np.float64(fc), fs=np.float64(fs), phase_offset=np.float64(phase_offset),
                  po_array=po_array, up=up, dn=dn, seed=seed, iq_crc=np.int64(int(iq.astype(np.int64).sum())),
                  x_idx=idx, deint_sub=x[idx], shift_sub=xs[idx], out_idx=oidx, out_sub=y[oidx],
                  out_len=y.shape[0], out_sum=np.complex128(y.sum()), out_absmax=np.float64(np.abs(y).max()),
                  shift_dtype=str(xs.dtype), out_dtype=str(y.dtype))
    if store_full:
        arrays.update(out=y)
    print(f"{name}: n={n} {kind} fc={fc} fs={fs} po={phase_offset} {up}/{dn} -> {y.shape[0]} {y.dtype} {dt:.2f}s")
    save(name, **arrays)


def resample_case(name, n, dtype, up, dn, profile="P1"):
    ref, _ = synth.make_frame(n, profile, 3)
    x = ref.astype(dtype)
    y = resample(x, up, dn)
    print(f"{name}: n={n} {dtype} {up}/{dn} -> {y.shape[0]} {y.dtype}")
    save(name, n=n, dtype=str(np.dtype(dtype)), up=up, dn=dn, profile=profile, out=y)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--big", action="store_true", help="also BASELINE config 2 (minutes, ~9 GB RAM)")
    ap.add_argument("--only", default=None)
    args = ap.parse_args()

    def want(name):
        return args.only is None or args.only in name

    # ---- shim proof: literal and shimmed reference on the same input
    if want("xambg_shim_proof"):
        ref, srv = synth.make_frame(8192, "P1")
        w = kaiser(8192)
        lit = fast_xambg(ref, srv, 20, 32, 8192, w)
        with fir_decimate_shim():
            shm = fast_xambg(ref, srv, 20, 32, 8192, w)
        lit2 = fast_xambg(ref, srv, 12, 16, 8192, None, False)
        with fir_decimate_shim():
            shm2 = fast_xambg(ref, srv, 12, 16, 8192, None, False)
        print("xambg_shim_proof: identical =", np.array_equal(lit, shm), np.array_equal(lit2, shm2))
        save("xambg_shim_proof", literal=lit, shim=shm, literal_long=lit2, shim_long=shm2)

    # ---- fast_xambg, literal reference, small and awkward shapes
    cases = [
        ("xambg_small_kaiser", dict(n=4096, F=32, R=20, profile="P1", window='kaiser', literal=True, input_len=4096)),
        ("xambg_small_nowin", dict(n=5000, F=16, R=33, profile="P0", window=None, literal=True)),
        ("xambg_pad_tuple", dict(n=4096, F=32, R=17, profile="P1", window='tuple', literal=True, input_len=4096, n_given=3000)),
        ("xambg_longfilt", dict(n=2048, F=16, R=10, profile="P1", window='kaiser', literal=True, input_len=2048, short_filt=False)),
        ("xambg_decim1", dict(n=64, F=64, R=5, profile="P0", window=None, literal=True)),
        ("xambg_decim2", dict(n=128, F=64, R=9, profile="P0", window='kaiser', literal=True, input_len=128)),
        ("xambg_odd_d251", dict(n=4016, F=16, R=25, profile="P1", window='kaiser', literal=True, input_len=4016)),
        ("xambg_even_d250", dict(n=4000, F=16, R=25, profile="P0", window=None, literal=True)),
        ("xambg_tail_ignored", dict(n=10000, F=32, R=40, profile="P1", window='kaiser', literal=True, input_len=10000)),
        ("xambg_r_ge_n", dict(n=96, F=8, R=130, profile="P0", window=None, literal=True)),
        ("xambg_nonpow2_F", dict(n=3000, F=24, R=12, profile="P1", window='kaiser', literal=True, input_len=3000)),
    ]
    for name, kw in cases:
        if want(name):
            xambg_case(name, **kw)

    # ---- BASELINE config 1 (200k, 64 x 100), shimmed reference
    if want("xambg_c1_p1"):
        xambg_case("xambg_c1_p1", n=200_000, F=64, R=100, profile="P1", window='kaiser', literal=False,
                   input_len=200_000, store_inputs=False)
    if want("xambg_c1_p0"):
        xambg_case("xambg_c1_p0", n=200_000, F=64, R=100, profile="P0", window=None, literal=False,
                   store_inputs=False)

    # ---- LS_Filter
    ls_cases = [
        ("ls_small", dict(n=4096, filter_len=20, reg=1.0, peek=10, profile="P1")),
        ("ls_small_peek0", dict(n=3000, filter_len=16, reg=0.5, peek=0, profile="P0")),
        ("ls_small_reg0", dict(n=2500, filter_len=12, reg=0.0, peek=3, profile="P1")),
        ("ls_mid", dict(n=50_000, filter_len=64, reg=1.0, peek=10, profile="P1", store_inputs=False)),
    ]
    for name, kw in ls_cases:
        if want(name):
            ls_case(name, **kw)
    if want("ls_c1_p1"):
        ls_case("ls_c1_p1", n=200_000, filter_len=100, reg=1.0, peek=10, profile="P1", store_inputs=False)
    if want("ls_c1_p0"):
        ls_case("ls_c1_p0", n=200_000, filter_len=100, reg=1.0, peek=10, profile="P0", store_inputs=False)

    # ---- LS_Filter_Toeplitz / LS_Filter_Multiple (what main.py:169-176 calls)
    if want("toep_small"):
        toeplitz_case("toep_small", n=4096, filter_len=20, peek=10, profile="P1")
    if want("toep_small_peek0"):
        toeplitz_case("toep_small_peek0", n=3000, filter_len=16, peek=0, profile="P0")
    if want("toep_mid"):
        toeplitz_case("toep_mid", n=262144, filter_len=175, peek=10, profile="P1", store_inputs=False)
    if want("multi_small"):
        multiple_case("multi_small", n=8192, filter_len=24, sample_rate=8192.0, bins=[0, 1, -1], profile="P1")
    if want("multi_fs_odd"):       # large phases at a non-power-of-two rate: pins numpy's reciprocal-multiply ramp
        multiple_case("multi_fs_odd", n=8192, filter_len=24, sample_rate=250000.0, bins=[0, 20000.5, -3000.25], profile="P1")
    if want("multi_main"):
        # the shipped PRconfig.yaml: half-CPI chunks of 262144 samples, 175 range cells, IF rate 2.4e6*13/119
        multiple_case("multi_main", n=262144, filter_len=175, sample_rate=2.4e6 * 13 / 119, bins=[0, 1, -1, 2, -2],
                      profile="P1", store_inputs=False)

    # ---- NLMS_filter
    if want("nlms_small"):
        nlms_case("nlms_small", n=6000, filter_len=30, mu=0.05, peek=10, profile="P1")
    if want("nlms_small_init"):
        nlms_case("nlms_small_init", n=5000, filter_len=24, mu=0.1, peek=4, profile="P1", with_init=True)
    if want("nlms_peek0"):
        nlms_case("nlms_peek0", n=3000, filter_len=17, mu=0.05, peek=0, profile="P0")
    if want("nlms_mid"):
        nlms_case("nlms_mid", n=20_000, filter_len=100, mu=0.05, peek=10, profile="P1")

    # ---- chained frame, config 1
    if want("frame_c1_p0"):
        frame_case("frame_c1_p0", 200_000, 64, 100, "P0", store_inputs=False)
    if want("frame_c1_p1"):
        frame_case("frame_c1_p1", 200_000, 64, 100, "P1", store_inputs=False)

    if args.big:
        if want("xambg_c2_p1"):
            xambg_case("xambg_c2_p1", n=2 ** 20, F=256, R=300, profile="P1", window='kaiser',
                       literal=False, input_len=2 ** 20, store_inputs=False)
        if want("ls_c2_p1"):
            ls_case("ls_c2_p1", n=2 ** 20, filter_len=300, reg=1.0, peek=10, profile="P1",
                    store_inputs=False)
        if want("frame_c2_p0"):
            frame_case("frame_c2_p0", 2 ** 20, 256, 300, "P0", store_inputs=False)

    # ---- rows either side of the hot path (SURVEY 8f): front end, CFAR, direct_xambg
    if want("cfar_main"):
        cfar_case("cfar_main", 256, 301, 18, 4)
    if want("cfar_thresh"):
        cfar_case("cfar_thresh", 64, 101, 18, 4, thresh=3.0)
    if want("cfar_odd"):
        cfar_case("cfar_odd", 40, 33, 9, 3)
    if want("cfar_tiny_map"):
        cfar_case("cfar_tiny_map", 12, 20, 18, 4)
    if want("direct_small"):
        direct_case("direct_small", 4096, 20, 16, 4096.0, "P1")
    if want("direct_odd"):
        direct_case("direct_odd", 5000, 33, 8, 250000.0, "P0")
    if want("direct_mid"):
        direct_case("direct_mid", 65536, 40, 32, 262144.0, "P1")
    if want("front_int8"):
        front_case("front_int8", 120_000, "int8", 300_000.0, 2_400_000.0, 1.2345, 13, 119)
    if want("front_int16_py"):
        front_case("front_int16_py", 50_001, "int16", -12345.678, 1_000_000.0, 0, 3, 2, po_array=False)
    if want("front_f32_short"):
        front_case("front_f32_short", 700, "float32", 10.0, 1000.0, 0.5, 13, 119)
    if want("front_chunk"):
        front_case("front_chunk", 9_600_000, "int8", 300_000.0, 2_400_000.0, 2.0 * np.pi * 7 * 0.125, 13, 119, store_full=False)
    if want("resample_c64"):
        resample_case("resample_c64", 30_000, np.complex64, 13, 119)
    if want("resample_c128"):
        resample_case("resample_c128", 9_000, np.complex128, 1, 4)


if __name__ == "__main__":
    main()
