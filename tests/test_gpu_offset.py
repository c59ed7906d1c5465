"""Channel alignment on the B200: find_channel_offset / offset_compensation / xcorr against the reference's arithmetic
(goldens made by running the reference, and oracle/offset_oracle.py, which makes the same SciPy calls).

Offsets must be exact.  Correlation values (the |xc| vector of find_channel_offset, every xcorr output) must be within
1e-6 of ||B1|| ||B2|| on every fixture and within 1e-5 of the peak where a delay is planted.  (SciPy's own FP32 FFT
correlation at P = 2^24 is 4.4e-8 of ||a|| ||b|| from float64.)"""
import ctypes as C
import threading

import numpy as np
import pytest

import passiveradar_b200 as prb
from passiveradar_b200 import _lib, synth
from oracle import offset_oracle as oo
import _golden as G
from conftest import record_parity

pytestmark = pytest.mark.gpu

OFFSET_GOLDENS = ["offset_int8_pos", "offset_c64_neg", "offset_nd4", "offset_zeros"]
XCORR_GOLDENS = [f"xcorr_{case}_{dt}" for case in ("equal", "s2_longer", "s1_longer", "lead_ne_lag")
                 for dt in ("c64", "c128", "f64")]


def norm_err(got, want, a, b):
    den = float(np.linalg.norm(np.asarray(a, np.complex128)) * np.linalg.norm(np.asarray(b, np.complex128)))
    return float(np.abs(np.asarray(got, np.complex128) - want).max() / den) if den else float(np.abs(got).max())


def peak_err(got, want):
    return float(np.abs(np.asarray(got, np.complex128) - want).max() / np.abs(want).max())


def check_offset_case(s1, s2, nd, nl, want_offset, want_xc, planted, tag):
    off, xc = prb.find_channel_offset(s1, s2, nd, nl, return_xc=True)
    assert isinstance(off, np.int64)
    assert off == want_offset, f"{tag}: offset {off} != {want_offset}"
    import scipy.signal as signal
    B1, B2 = signal.decimate(s1, nd), signal.decimate(s2, nd)
    e_norm = norm_err(xc, want_xc, B1, B2)
    assert e_norm <= 1e-6, f"{tag}: |xc| error {e_norm:.2e} of ||B1|| ||B2||"
    figures = {"offset": int(off), "xc_vs_ref_norm": e_norm}
    if planted:
        e_peak = peak_err(xc, want_xc)
        assert e_peak <= 1e-5, f"{tag}: |xc| error {e_peak:.2e} of the peak"
        figures["xc_vs_ref_peak"] = e_peak
    record_parity(f"offset_{tag}", **figures)
    return off, xc


@pytest.mark.parametrize("name", OFFSET_GOLDENS)
def test_offset_goldens(name):
    g = G.load(name)
    s1, s2 = g["s1"], g["s2"]
    check_offset_case(s1, s2, int(g["nd"]), int(g["nl"]), int(g["offset"]), g["xc"], name != "offset_zeros", name)


def test_offset_main_shape_golden():
    """main.py's call on the default config's int8 channels (5 242 880 entries, nl = 5e6); inputs regenerated."""
    g = G.load("offset_main")
    s1, s2 = synth.offset_pair(int(g["n"]), int(g["planted"]), str(g["kind"]), int(g["seed"]))
    np.testing.assert_array_equal(s1[::100003], g["s1_probe"])
    off, xc = prb.find_channel_offset(s1, s2, int(g["nd"]), int(g["nl"]), return_xc=True)
    assert off == int(g["offset"]) == int(g["planted"])
    top2 = np.sort(xc)[-2:][::-1]
    np.testing.assert_allclose(top2, g["top2"], rtol=1e-5)
    sub = xc[::int(g["stride"])]
    assert float(np.abs(sub - g["xc_sub"]).max() / g["top2"][0]) <= 1e-5
    record_parity("offset_main_golden", offset=int(off), top_rel=float(abs(top2[0] - g["top2"][0]) / g["top2"][0]))


def test_zero_input_tie_gives_first_lag():
    z = np.zeros(5000, np.int8)
    for nd in (1, 4):
        assert prb.find_channel_offset(z, z, nd, 300) == -300 * nd


@pytest.mark.parametrize("kind,planted,nd", [("complex64", -37, 1), ("int8", 123, 1), ("int16", 5, 1),
                                             ("complex64", 48, 4), ("int8", -400, 4), ("complex64", 0, 10)])
def test_offset_matches_oracle_small(kind, planted, nd):
    s1, s2 = synth.offset_pair(40000, planted, kind)
    want, want_xc = oo.channel_offset_oracle(s1, s2, nd, 700)
    assert want == planted
    check_offset_case(s1, s2, nd, 700, want, want_xc, True, f"small_{kind}_{planted}_{nd}")


def test_offset_unequal_lengths_and_short_window():
    s1, s2 = synth.offset_pair(30000, 11, "complex64")
    for a, b, nl in ((s1, s2[:20000], 500), (s1[:20000], s2, 500), (s1, s2[:1000], 10)):
        want, want_xc = oo.channel_offset_oracle(a, b, 1, nl)
        off, xc = prb.find_channel_offset(a, b, 1, nl, return_xc=True)
        assert off == want and xc.shape == want_xc.shape


@pytest.mark.parametrize("name", XCORR_GOLDENS)
def test_xcorr_goldens(name):
    g = G.load(name)
    s1, s2 = g["s1"], g["s2"]
    out = prb.xcorr(s1, s2, int(g["nlead"]), int(g["nlag"]))
    assert out.dtype == g["out"].dtype and out.shape == g["out"].shape
    e = norm_err(out, g["out"], s1, s2)
    assert e <= 1e-6, f"{name}: {e:.2e}"
    record_parity(name, vs_ref_norm=e)


def test_xcorr_dtypes_and_planted_peak():
    s1, s2 = synth.offset_pair(50000, 250, "complex64")
    for dt in (np.complex64, np.complex128, np.float32, np.float64):
        a = s1.astype(dt) if np.dtype(dt).kind == 'c' else s1.real.astype(dt)
        b = s2.astype(dt) if np.dtype(dt).kind == 'c' else s2.real.astype(dt)
        want = oo.xcorr_oracle(a, b, 3000, 1000)
        got = prb.xcorr(a, b, 3000, 1000)
        assert got.dtype == want.dtype and got.shape == want.shape
        assert norm_err(got, want, a, b) <= 1e-6
        assert peak_err(got, want) <= 1e-5
        assert np.argmax(np.abs(got)) == np.argmax(np.abs(want))


def test_offset_compensation():
    x1, x2 = synth.offset_pair(60000, 29, "complex64")
    y = prb.offset_compensation(x1, x2, 40000, 1, 200)
    np.testing.assert_array_equal(y, oo.offset_compensation_oracle(x1, x2, 40000, 1, 200))
    same = prb.offset_compensation(x1, x1.copy(), 40000, 1, 200)
    assert same is not x1 and np.array_equal(same, x1)
    x3 = x1.copy()
    assert prb.offset_compensation(x1, x3, 40000, 1, 200) is x3          # offset 0: x2 itself


def test_device_pointer_path_is_bit_identical():
    import torch
    s1, s2 = synth.offset_pair(100000, -77, "int8")
    nd, nl = 2, 3000
    off, xc = prb.find_channel_offset(s1, s2, nd, nl, return_xc=True)
    from passiveradar_b200.signal_utils import _decimate_sos
    sos, _ = _decimate_sos(nd, False)
    dev = _lib.current_device()
    t1 = torch.from_numpy(s1).cuda(dev)
    t2 = torch.from_numpy(s2).cuda(dev)
    doff = torch.zeros(1, dtype=torch.int64, device=f"cuda:{dev}")
    dxc = torch.empty(xc.shape[0], dtype=torch.float32, device=f"cuda:{dev}")
    stream = torch.cuda.current_stream(dev)
    lib = _lib.load()
    _lib.check(lib.prc_channel_offset(t1.data_ptr(), s1.shape[0], t2.data_ptr(), s2.shape[0], _lib.SIG_I8, nd, nl,
                                      sos.ctypes.data, sos.shape[0], doff.data_ptr(), dxc.data_ptr(),
                                      _lib.MEM_DEVICE, dev, C.c_void_p(stream.cuda_stream), 0))
    assert int(doff.item()) == off
    assert np.array_equal(dxc.cpu().numpy(), xc)
    # xcorr on device pointers
    a, b = synth.offset_pair(20000, 5, "complex64")
    host = prb.xcorr(a, b, 100, 200)
    ta, tb = torch.from_numpy(a).cuda(dev), torch.from_numpy(b).cuda(dev)
    tout = torch.empty(host.shape[0], dtype=torch.complex64, device=f"cuda:{dev}")
    lag0, nlags = 20000 - 20000 + 100, 20000 + 300 - 20000 + 1
    _lib.check(lib.prc_xcorr_c64(ta.data_ptr(), 20000, tb.data_ptr(), 20000, lag0, nlags, tout.data_ptr(),
                                 _lib.MEM_DEVICE, dev, C.c_void_p(stream.cuda_stream), 0))
    assert np.array_equal(tout.cpu().numpy(), host)


def test_concurrent_threads_match_serial_calls():
    pairs = [synth.offset_pair(60000, d, k, seed=100 + i)
             for i, (d, k) in enumerate([(13, "int8"), (-90, "complex64"), (400, "int16"), (-5, "complex64")])]
    serial = [prb.find_channel_offset(a, b, 1, 2000, return_xc=True) for a, b in pairs]
    results = [None] * len(pairs)

    def work(i):
        results[i] = prb.find_channel_offset(pairs[i][0], pairs[i][1], 1, 2000, return_xc=True)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(pairs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for (o1, x1), (o2, x2) in zip(serial, results):
        assert o1 == o2 and np.array_equal(x1, x2)


def test_argument_errors_are_invalid():
    lib = _lib.load()
    sos = np.zeros((4, 6))
    x = np.zeros(100, np.complex64)
    off = np.zeros(1, np.int64)
    st = lib.prc_channel_offset(x.ctypes.data, 100, x.ctypes.data, 100, _lib.SIG_C64, 1, 10, sos.ctypes.data, 4,
                                off.ctypes.data, None, _lib.MEM_HOST, _lib.current_device(), None, 0)
    assert st == _lib.PRC_E_INVALID                       # sos[:, 3] != 1
    st = lib.prc_xcorr_c64(x.ctypes.data, 100, x.ctypes.data, 100, 0, 0, x.ctypes.data, _lib.MEM_HOST,
                           _lib.current_device(), None, 0)
    assert st == _lib.PRC_E_INVALID


# ---- the shapes main.py runs (oracle inside the test) --------------------------------------------------------------
SHAPES = [("int8", 5242880, 1234), ("complex64", 2621440, -2345), ("int8", 10485760, 777)]


@pytest.mark.slow
@pytest.mark.parametrize("kind,n,planted", SHAPES, ids=["int8_main", "c64_interleaved", "int8_tiled"])
def test_main_shapes(kind, n, planted):
    nl = 5000000
    s1, s2 = synth.offset_pair(n, planted, kind)
    want, want_xc = oo.channel_offset_oracle(s1, s2, 1, nl)
    assert want == planted
    check_offset_case(s1, s2, 1, nl, want, want_xc, True, f"shape_{kind}_{n}")
