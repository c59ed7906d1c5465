"""Pins the CPU oracle to the reference: every oracle function must reproduce the
outputs the reference's own code produced (tests/golden/*.npz, made by
tests/golden/make_golden.py with /root/reference on the path)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import _golden as G
from oracle import clutter_oracle as co
from oracle import xambg_oracle as xo


def test_shim_is_bit_identical_to_literal_reference():
    g = G.load("xambg_shim_proof")
    assert np.array_equal(g["literal"], g["shim"])
    assert np.array_equal(g["literal_long"], g["shim_long"])


@pytest.mark.parametrize("name", G.XAMBG_SMALL + G.XAMBG_C1)
def test_xambg_oracle_matches_reference(name):
    g = G.load(name)
    ref, srv = G.inputs(g)
    R, F, input_len, window, short = G.xambg_args(g)
    out = xo.fast_xambg_oracle(ref, srv, R, F, input_len, window, short)
    assert out.shape == g["out"].shape and out.dtype == np.complex64
    # same library calls on the same data: bit-identical, not merely close
    assert np.array_equal(out, g["out"]), G.rel_inf(out, g["out"])


@pytest.mark.parametrize("name", G.XAMBG_SMALL + ["xambg_c1_p1"])
def test_xambg_truth_formula_matches_reference(name):
    g = G.load(name)
    ref, srv = G.inputs(g)
    R, F, input_len, window, short = G.xambg_args(g)
    truth = xo.fast_xambg_truth(ref, srv, R, F, input_len, window, short)
    assert G.rel_inf(g["out"], truth) < 2e-6


_LS_ORACLE_RUN = """
import sys
import numpy as np
sys.path[:0] = sys.argv[1:3]
import _golden as G
from oracle import clutter_oracle as co
g = G.load(sys.argv[3])
ref, srv = G.inputs(g)
out, taps = co.ls_filter_oracle(ref, srv, int(g["filter_len"]), float(g["reg"]), int(g["peek"]), True)
np.savez(sys.argv[4], out=out, taps=taps)
"""


@pytest.mark.parametrize("name", G.LS_SMALL + G.LS_C1)
def test_ls_oracle_matches_reference(name, tmp_path):
    # the complex64 Gram of LS_Filter is one cgemm over n samples; its rounding depends on the BLAS kernels and thread
    # count (up to 1e-5 in the taps of a 200k-sample frame), so the oracle runs with the BLAS the goldens were made with
    res = tmp_path / "ls.npz"
    tests_dir = os.path.dirname(os.path.abspath(__file__))
    subprocess.run([sys.executable, "-c", _LS_ORACLE_RUN, tests_dir, os.path.dirname(tests_dir), name, str(res)],
                   env=dict(os.environ, **G.GOLDEN_BLAS), check=True, timeout=600)
    g = G.load(name)
    with np.load(res) as z:
        out, taps = z["out"], z["taps"]
    assert out.dtype == np.complex64 and taps.dtype == np.complex64
    # BLAS threading may reorder the cgemm reduction between runs: allow float32 noise only
    assert G.rel_inf(taps, g["taps"]) < 2e-6
    assert G.rel_inf(out[g["out_idx"]], g["out_sub"], den=float(g["srv_absmax"])) < 2e-6


@pytest.mark.parametrize("name", G.LS_SMALL)
def test_ls_truth_close_to_reference(name):
    g = G.load(name)
    ref, srv = G.inputs(g)
    out, taps = co.ls_filter_truth(ref, srv, int(g["filter_len"]), float(g["reg"]), int(g["peek"]))
    assert G.rel_inf(g["taps"], taps) < 2e-5
    assert G.rel_inf(g["out_sub"], out[g["out_idx"]], den=float(g["srv_absmax"])) < 2e-5


@pytest.mark.parametrize("name", G.NLMS_ALL)
def test_nlms_oracle_matches_reference(name):
    g = G.load(name)
    init = g["init"] if g["init"].shape[0] else None
    out, w = co.nlms_filter_oracle(g["ref"], g["srv"], int(g["filter_len"]), float(g["mu"]),
                                   int(g["peek"]), init, True)
    assert np.array_equal(out, g["out"]) or G.rel_inf(out, g["out"]) < 1e-6
    assert G.rel_inf(w, g["taps"]) < 1e-6
    fl = int(g["filter_len"]) if init is None else init.shape[0] - int(g["peek"])
    assert not out[:fl].any()
    if int(g["peek"]):
        assert not out[-int(g["peek"]):].any()


@pytest.mark.parametrize("name", ["nlms_small", "nlms_small_init"])
def test_nlms_truth_close_to_reference(name):
    g = G.load(name)
    init = g["init"] if g["init"].shape[0] else None
    out, w = co.block_nlms_truth(g["ref"], g["srv"], int(g["filter_len"]), float(g["mu"]),
                                 int(g["peek"]), 1, init)
    assert G.rel_inf(g["out"], out) < 1e-5
    assert G.rel_inf(g["taps"], w) < 1e-4


def test_block_nlms_block1_is_nlms_and_blocks_differ():
    g = G.load("nlms_small")
    a = co.block_nlms_oracle(g["ref"], g["srv"], int(g["filter_len"]), float(g["mu"]), int(g["peek"]), 1)
    assert np.array_equal(a, g["out"]) or G.rel_inf(a, g["out"]) < 1e-6
    b, wb = co.block_nlms_oracle(g["ref"], g["srv"], int(g["filter_len"]), float(g["mu"]), int(g["peek"]),
                                 16, None, True)
    t, wt = co.block_nlms_truth(g["ref"], g["srv"], int(g["filter_len"]), float(g["mu"]), int(g["peek"]), 16)
    assert G.rel_inf(b, t) < 1e-5
    assert G.rel_inf(b, g["out"]) > 1e-4        # a genuinely different algorithm for B > 1


def test_frame_chain_goldens_consistent_with_oracle():
    g = G.load("frame_c1_p0")
    ref, srv = G.inputs(g)
    cleaned = co.ls_filter_oracle(ref, srv, int(g["R"]))
    import scipy.signal as signal
    out = xo.fast_xambg_oracle(ref, cleaned, int(g["R"]), int(g["F"]), int(g["n"]),
                               signal.get_window(("kaiser", 5.0), int(g["n"])))
    assert G.rel_inf(out, g["out"]) < 1e-5


def test_shape_mismatch_raises_like_reference():
    a = np.zeros(10, np.complex64)
    b = np.zeros(11, np.complex64)
    with pytest.raises(ValueError, match="same length"):
        xo.fast_xambg_oracle(a, b, 2, 2)
    with pytest.raises(ValueError, match="same length"):
        co.ls_filter_oracle(a, b, 2)


@pytest.mark.parametrize("name", G.NLMS_ALL)
def test_c_nlms_oracle_matches_reference(name):
    g = G.load(name)
    init = g["init"] if g["init"].shape[0] else None
    out, w = co.block_nlms_oracle_c(g["ref"], g["srv"], int(g["filter_len"]), float(g["mu"]),
                                    int(g["peek"]), 1, init)
    assert G.rel_inf(out, g["out"]) < 2e-6
    assert G.rel_inf(w, g["taps"]) < 2e-5


def test_c_block_nlms_matches_python_definition():
    g = G.load("nlms_small")
    a, wa = co.block_nlms_oracle_c(g["ref"], g["srv"], int(g["filter_len"]), float(g["mu"]), int(g["peek"]), 16)
    b, wb = co.block_nlms_oracle(g["ref"], g["srv"], int(g["filter_len"]), float(g["mu"]), int(g["peek"]), 16,
                                 None, True)
    assert G.rel_inf(a, b) < 2e-6 and G.rel_inf(wa, wb) < 2e-5


@pytest.mark.parametrize("name", G.TOEP_ALL)
def test_toeplitz_oracle_matches_reference(name):
    g = G.load(name)
    ref, srv = G.inputs(g)
    out, taps = co.ls_filter_toeplitz_oracle(ref, srv, int(g["filter_len"]), int(g["peek"]), True)
    assert out.dtype == np.complex128 and taps.dtype == np.complex128
    assert G.rel_inf(taps, g["taps"]) < 1e-9
    assert G.rel_inf(out[g["out_idx"]], g["out_sub"], den=float(g["srv_absmax"])) < 1e-9


@pytest.mark.parametrize("name", G.MULTI_ALL)
def test_multiple_oracle_matches_reference(name):
    g = G.load(name)
    ref, srv = G.inputs(g)
    out = co.ls_filter_multiple_oracle(ref, srv, int(g["filter_len"]), float(g["sample_rate"]), list(g["bins"]))
    assert G.rel_inf(out[g["out_idx"]], g["out_sub"], den=float(g["srv_absmax"])) < 1e-9
    sh = co.frequency_shift_oracle(ref, float(g["bins"][-1]), float(g["sample_rate"]))
    assert np.array_equal(sh[g["out_idx"]], g["shift_sample"])


@pytest.mark.parametrize("name", ["nlms_small", "nlms_peek0"])
@pytest.mark.parametrize("L", [8, 32])
def test_block_exact_nlms_is_the_reference_recurrence(name, L):
    """The triangular-system form nlms_block_kernel evaluates equals the reference's sample-serial NLMS
    (golden produced by the reference) up to complex64 round-off."""
    g = G.load(name)
    ref, srv = G.inputs(g)
    out, taps = co.nlms_block_exact(ref, srv, int(g["filter_len"]), float(g["mu"]), int(g["peek"]), L)
    den = np.abs(srv).max()
    assert np.abs(out - g["out"]).max() / den <= 2e-6
    assert np.abs(taps - g["taps"]).max() / np.abs(g["taps"]).max() <= 5e-6
