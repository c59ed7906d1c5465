"""Helpers shared by the parity tests: load goldens, rebuild their seeded inputs."""
import os

import numpy as np
import scipy.signal as signal

from passiveradar_b200 import synth

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# OpenBLAS configuration the goldens were made with (make_golden.py sets it): complex64 matrix products of the
# reference round differently with other kernels or thread counts
GOLDEN_BLAS = {"OPENBLAS_CORETYPE": "SkylakeX", "OPENBLAS_NUM_THREADS": "8"}


def load(name):
    path = os.path.join(GOLDEN_DIR, name + ".npz")
    with np.load(path, allow_pickle=False) as z:
        return {k: z[k] for k in z.files}


def have(name):
    return os.path.exists(os.path.join(GOLDEN_DIR, name + ".npz"))


def inputs(g):
    """(ref, srv) of a golden: stored arrays when present, else regenerated from the seed
    and checked against the stored fingerprint (guards against RNG-stream drift)."""
    if "ref" in g:
        return g["ref"], g["srv"]
    ref, srv = synth.make_frame(int(g["n"]), str(g["profile"]), int(g["frame"]))
    np.testing.assert_array_equal(synth.frame_digest(ref, srv), g["digest"])
    return ref, srv


def xambg_args(g):
    """Positional args (after ref, srv) the golden was generated with."""
    n = int(g["n"])
    input_len = None if int(g["input_len"]) < 0 else int(g["input_len"])
    nn = n if input_len is None else input_len
    w = str(g["window"])
    if w == "kaiser":
        window = signal.get_window(("kaiser", 5.0), nn)
    elif w == "tuple":
        window = ("kaiser", 5.0)
    else:
        window = None
    return int(g["R"]), int(g["F"]), input_len, window, bool(g["short_filt"])


def rel_inf(a, b, den=None):
    a = np.asarray(a)
    b = np.asarray(b)
    d = np.abs(b).max() if den is None else den
    return float(np.abs(a - b).max() / d)


XAMBG_SMALL = ["xambg_small_kaiser", "xambg_small_nowin", "xambg_pad_tuple", "xambg_longfilt",
               "xambg_decim1", "xambg_decim2", "xambg_odd_d251", "xambg_even_d250",
               "xambg_tail_ignored", "xambg_r_ge_n", "xambg_nonpow2_F"]
XAMBG_C1 = ["xambg_c1_p1", "xambg_c1_p0"]
LS_SMALL = ["ls_small", "ls_small_peek0", "ls_small_reg0", "ls_mid"]
LS_C1 = ["ls_c1_p1", "ls_c1_p0"]
NLMS_ALL = ["nlms_small", "nlms_small_init", "nlms_peek0", "nlms_mid"]

TOEP_ALL = ["toep_small", "toep_small_peek0", "toep_mid"]
MULTI_ALL = ["multi_small", "multi_fs_odd", "multi_main"]


CFAR_ALL = ["cfar_main", "cfar_thresh", "cfar_odd", "cfar_tiny_map"]
DIRECT_ALL = ["direct_small", "direct_odd", "direct_mid"]
FRONT_SMALL = ["front_int8", "front_int16_py", "front_f32_short"]
FRONT_BIG = ["front_chunk"]
RESAMPLE_ALL = ["resample_c64", "resample_c128"]


def front_inputs(g):
    """(iq, fc, fs, phase_offset as the golden passed it, up, dn) of a front-end golden."""
    iq = synth.raw_iq(int(g["n"]), str(g["kind"]), int(g["seed"]))
    assert int(iq.astype(np.int64).sum()) == int(g["iq_crc"]) or str(g["kind"]) == "float32"
    po = float(g["phase_offset"])
    po = np.array([po]) if bool(g["po_array"]) else (int(po) if po == int(po) else po)
    return iq, float(g["fc"]), float(g["fs"]), po, int(g["up"]), int(g["dn"])
