"""Host-side checks of the channel-alignment drop-ins (find_channel_offset, offset_compensation, xcorr): the oracle
against the reference's goldens, numpy models of the device algorithms (chunked zero-phase IIR, tile plan of the
long-lag correlation), argument errors before any device call, install().  No GPU needed."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.signal as signal

import passiveradar_b200 as prb
from passiveradar_b200 import _lib, signal_utils
from oracle import offset_oracle as oo
import _golden as G

OFFSET_GOLDENS = ["offset_int8_pos", "offset_c64_neg", "offset_nd4", "offset_zeros"]
XCORR_GOLDENS = [f"xcorr_{case}_{dt}" for case in ("equal", "s2_longer", "s1_longer", "lead_ne_lag")
                 for dt in ("c64", "c128", "f64")]
REFERENCE = os.environ.get("PR_REFERENCE", "/root/reference")


# ---- oracle == reference ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", OFFSET_GOLDENS)
def test_oracle_equals_offset_goldens(name):
    g = G.load(name)
    off, xc = oo.channel_offset_oracle(g["s1"], g["s2"], int(g["nd"]), int(g["nl"]))
    assert off == int(g["offset"])
    np.testing.assert_array_equal(xc, g["xc"])
    if name != "offset_zeros":
        assert int(g["offset"]) == int(g["planted"])
    else:
        assert int(g["offset"]) == -int(g["nl"]) * int(g["nd"])          # all-zero |xc|: the first lag wins


@pytest.mark.parametrize("name", XCORR_GOLDENS)
def test_oracle_equals_xcorr_goldens(name):
    g = G.load(name)
    out = oo.xcorr_oracle(g["s1"], g["s2"], int(g["nlead"]), int(g["nlag"]))
    assert out.dtype == g["out"].dtype
    np.testing.assert_array_equal(out, g["out"])


@pytest.mark.parametrize("name", ["offcomp_zero", "offcomp_shift"])
def test_oracle_equals_offset_compensation_goldens(name):
    g = G.load(name)
    out = oo.offset_compensation_oracle(g["x1"], g["x2"], int(g["ns"]), int(g["ndec"]), int(g["nlag"]))
    np.testing.assert_array_equal(out, g["out"])
    assert bool(g["same"]) == (name == "offcomp_zero")


def test_main_shape_golden_inputs_regenerate():
    g = G.load("offset_main")
    from passiveradar_b200 import synth
    s1, _ = synth.offset_pair(int(g["n"]), int(g["planted"]), str(g["kind"]), int(g["seed"]))
    np.testing.assert_array_equal(s1[::100003], g["s1_probe"])
    assert s1.shape[0] == 5242880 and s1.dtype == np.int8 and int(g["offset"]) == int(g["planted"])


@pytest.mark.skipif(not os.path.isdir(os.path.join(REFERENCE, "passiveRadar")), reason="reference tree not available")
@pytest.mark.parametrize("name", ["offset_nd4", "xcorr_s1_longer_c64"])
def test_committed_offset_golden_is_what_the_reference_produces(name, tmp_path):
    env = dict(os.environ, PR_GOLDEN_OUT=str(tmp_path), PR_REFERENCE=REFERENCE)
    script = os.path.join(G.GOLDEN_DIR, "make_golden_offset.py")
    subprocess.run([sys.executable, script, "--only", name], check=True, env=env, capture_output=True, timeout=600)
    committed = G.load(name)
    with np.load(tmp_path / (name + ".npz"), allow_pickle=False) as z:
        fresh = {k: z[k] for k in z.files}
    assert set(fresh) == set(committed)
    for k in committed:
        if k != "seconds":
            np.testing.assert_array_equal(fresh[k], committed[k], err_msg=f"{name}[{k}]")


# ---- numpy model of the device's zero-phase IIR (csrc/xcorr.cuh, iir_fwd_kernel / iir_bwd_kernel) -------------------
def warm_length(sos):
    rho = max(abs(p) for s in sos for p in np.roots(s[3:]))
    return max(32, math.ceil(math.log(1e-20) / math.log(rho)))


def chunked_sosfilt(sos, x, zi0, chunk, warm):
    """What one thread per chunk computes: zero state `warm` samples before its chunk, exact state at the start."""
    y = np.empty_like(x)
    zero = np.zeros((sos.shape[0], 2), dtype=x.dtype)
    for j0 in range(0, x.shape[0], chunk):
        j1 = min(j0 + chunk, x.shape[0])
        js = j0 - warm
        if js <= 0:
            seg, _ = signal.sosfilt(sos, x[0:j1], zi=zi0 * x[0])
            y[j0:j1] = seg[j0:]
        else:
            seg, _ = signal.sosfilt(sos, x[js:j1], zi=zero)
            y[j0:j1] = seg[j0 - js:]
    return y


@pytest.mark.parametrize("nd,dtype", [(1, np.float64), (4, np.complex128), (10, np.float64)])
def test_chunked_iir_model_equals_sosfiltfilt(nd, dtype):
    rng = np.random.default_rng(nd)
    n = 30000
    x = rng.standard_normal(n) + (1j * rng.standard_normal(n) if dtype == np.complex128 else 0)
    sos = signal.cheby1(8, 0.05, 0.8 / nd, output='sos')
    warm = warm_length(sos)
    assert warm >= 1000
    P = 27
    ext = np.concatenate([2 * x[:1] - x[P:0:-1], x, 2 * x[-1:] - x[-2:-P - 2:-1]])
    zi = signal.sosfilt_zi(sos)
    yf = chunked_sosfilt(sos, ext, zi, 1024, warm)
    yb = chunked_sosfilt(sos, yf[::-1].copy(), zi, 1024, warm)[::-1]
    got = yb[P:-P][::nd]
    want = signal.decimate(x, nd)
    assert np.abs(got - want).max() / np.abs(want).max() <= 1e-12


# ---- tile plan of the long-lag correlation (prcore.cu xc_plan) ------------------------------------------------------
def xc_plan(nx, nlags, pmin=1 << 20, pmax=1 << 24):
    need = nx + nlags - 1
    if need <= pmax:
        P = pmin
        while P < need:
            P <<= 1
        seg, tile = nx, nlags
    else:
        P = pmax
        tile = min(nlags, pmax // 2)
        seg = pmax - tile + 1
        if nx < seg:
            seg, tile = nx, pmax - nx + 1
    return P, seg, tile, -(-nx // seg), -(-nlags // tile)


def tiled_correlation(x, y, lag0, nlags, pmin, pmax):
    """float64 circular FFTs exactly as the device tiles them; returns out and how often each lag was written."""
    P, seg, tile, nseg, ntile = xc_plan(x.shape[0], nlags, pmin, pmax)
    assert seg + min(tile, nlags) - 1 <= P                 # no circular wrap inside a tile
    out = np.zeros(nlags, np.complex128)
    hits = np.zeros(nlags, np.int64)
    for ti in range(ntile):
        j0 = ti * tile
        nt = min(tile, nlags - j0)
        m_lo = lag0 - j0 - nt + 1
        S = np.zeros(P, np.complex128)
        for si in range(nseg):
            s = si * seg
            xs = np.zeros(P, np.complex128)
            xs[:min(seg, x.shape[0] - s)] = x[s:s + seg]
            idx = s + m_lo + np.arange(P)
            ys = np.where((idx >= 0) & (idx < y.shape[0]), y[np.clip(idx, 0, y.shape[0] - 1)], 0)
            S += np.fft.fft(xs) * np.conj(np.fft.fft(ys))
        circ = np.fft.fft(S) / P                           # forward DFT of X conj(Y): sum_i x[i] conj(y[i + m])
        m = np.arange(nt)
        out[j0 + nt - 1 - m] = circ[m]
        hits[j0 + nt - 1 - m] += 1
    return out, hits


@pytest.mark.parametrize("n1,n2,nl,nd", [(200, 200, 300, 1), (700, 300, 40, 1), (300, 700, 40, 2), (1000, 1000, 900, 1),
                                         (5000, 40, 2, 1), (64, 64, 0, 1), (900, 900, 1000, 3)])
def test_tile_plan_covers_every_lag_once_without_aliasing(n1, n2, nl, nd):
    rng = np.random.default_rng(n1 + n2 + nl)
    x = rng.standard_normal(-(-n1 // nd)) + 1j * rng.standard_normal(-(-n1 // nd))
    y = rng.standard_normal(-(-n2 // nd)) + 1j * rng.standard_normal(-(-n2 // nd))
    lag0, nlags = signal_utils._xcorr_window(x.shape[0], y.shape[0], nl, nl)
    got, hits = tiled_correlation(x, y, lag0, nlags, pmin=64, pmax=256)       # scaled-down P: tiles and segments
    assert np.all(hits == 1)
    want = oo.xcorr_oracle(x, y, nl, nl)
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-9 * np.abs(want).max())


@pytest.mark.parametrize("n,nl", [(5242880, 5000000), (2621440, 5000000), (10485760, 5000000), (1000, 5000000),
                                  (40_000_000, 100), (30_000, 3_000)])
def test_tile_plan_at_full_size(n, nl):
    lag0, nlags = signal_utils._xcorr_window(n, n, nl, nl)
    P, seg, tile, nseg, ntile = xc_plan(n, nlags)
    assert seg + tile - 1 <= P <= 1 << 24 and seg * nseg >= n and tile * ntile >= nlags
    if n + nlags - 1 <= 1 << 24:
        assert nseg == ntile == 1                          # main.py's default shape is one transform
    if n == 10485760:
        assert nseg == 2 and ntile == 2                    # cpi_seconds_nominal: 4 needs tiling


# ---- interface ------------------------------------------------------------------------------------------------------
def positional(f):
    import inspect
    return [(p.name, p.default) for p in inspect.signature(f).parameters.values() if p.kind == p.POSITIONAL_OR_KEYWORD]


def test_signatures_and_defaults_match_the_reference():
    import inspect
    E = inspect.Parameter.empty
    assert positional(prb.find_channel_offset) == [("s1", E), ("s2", E), ("nd", E), ("nl", E)]
    assert positional(prb.offset_compensation) == [("x1", E), ("x2", E), ("ns", E), ("ndec", E), ("nlag", 2000)]
    assert positional(prb.xcorr) == [("s1", E), ("s2", E), ("nlead", E), ("nlag", E)]
    for name in ("xcorr", "find_channel_offset", "offset_compensation"):
        assert name in prb.__all__


@pytest.fixture
def no_device(monkeypatch):
    """Any library call fails the test: argument errors must come first."""
    def boom(*a, **k):
        raise AssertionError("the library was called")
    monkeypatch.setattr(_lib, "load", boom)


def test_reference_exceptions_before_any_device_call(no_device):
    x = np.zeros(1000, np.int8)
    short = np.zeros(27, np.int8)
    with pytest.raises(ValueError, match="padlen"):
        prb.find_channel_offset(short, x, 1, 10)
    with pytest.raises(ValueError, match="padlen"):
        prb.find_channel_offset(x, short, 1, 10)
    with pytest.raises(ZeroDivisionError):
        prb.find_channel_offset(x, x, 0, 10)
    with pytest.raises(ValueError):
        prb.find_channel_offset(x, x, -2, 10)
    with pytest.raises(TypeError):
        prb.find_channel_offset(x, x, 1.5, 10)
    with pytest.raises(ValueError):
        prb.find_channel_offset(x, x, 1, -1)
    c = np.zeros(100, np.complex64)
    with pytest.raises(TypeError):
        prb.xcorr(np.zeros(100, np.int16), c, 1, 1)
    with pytest.raises(ValueError):
        prb.xcorr(c, c, -1, 1)
    with pytest.raises(ValueError):
        prb.offset_compensation(short, short, 27, 1)


def test_reference_raises_the_same_exception_types():
    import scipy.signal as s
    x = np.zeros(1000, np.int8)
    with pytest.raises(ValueError):
        s.sosfiltfilt(s.cheby1(8, 0.05, 0.8, output='sos'), np.zeros(27))
    with pytest.raises(ZeroDivisionError):
        s.decimate(x, 0)
    with pytest.raises(ValueError):
        s.decimate(x, -2)
    with pytest.raises(TypeError):
        s.decimate(x, 1.5)
    with pytest.raises(ValueError):
        np.pad(np.zeros(10), (-1, -1))


def test_without_a_device_there_is_no_cpu_fallback():
    if _lib.device_count() > 0:
        pytest.skip("a CUDA device is present")
    x = np.zeros(1000, np.int8)
    with pytest.raises(_lib.PrcoreError):
        prb.find_channel_offset(x, x, 1, 10)
    c = np.ones(100, np.complex64)
    with pytest.raises(_lib.PrcoreError):
        prb.xcorr(c, c, 5, 5)
    with pytest.raises(_lib.PrcoreError):
        prb.offset_compensation(c, c, 100, 1, 5)


def test_install_swaps_channel_alignment_but_not_xcorr(tmp_path, monkeypatch):
    pkg = tmp_path / "fakeRadar2"
    pkg.mkdir()
    (pkg / "__init__.py").write_text("")
    (pkg / "range_doppler_processing.py").write_text("def fast_xambg(*a, **k):\n    return 'cpu'\n")
    (pkg / "clutter_removal.py").write_text("def LS_Filter(*a, **k):\n    return 'cpu'\n")
    (pkg / "signal_utils.py").write_text(
        "def find_channel_offset(*a, **k):\n    return 'cpu'\n"
        "def offset_compensation(*a, **k):\n    return 'cpu'\n"
        "def xcorr(*a, **k):\n    return 'untouched'\n")
    monkeypatch.syspath_prepend(str(tmp_path))
    replaced = prb.install("fakeRadar2")
    from fakeRadar2.signal_utils import find_channel_offset, offset_compensation, xcorr
    assert find_channel_offset is prb.find_channel_offset and offset_compensation is prb.offset_compensation
    assert xcorr() == "untouched"
    assert "fakeRadar2.signal_utils.find_channel_offset" in replaced
    for m in [k for k in sys.modules if k.startswith("fakeRadar2")]:
        del sys.modules[m]
