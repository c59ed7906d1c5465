#!/usr/bin/env python
"""Generate the channel-alignment goldens under tests/golden/ by EXECUTING THE REFERENCE.

Run where a copy of the reference is available (PR_REFERENCE, default /root/reference):

    python tests/golden/make_golden_offset.py [--only NAME]

Every stored output comes from the reference's own ``passiveRadar.signal_utils.{find_channel_offset,
offset_compensation, xcorr}`` (signal_utils.py:29-78; main.py:54, :83).  ``find_channel_offset`` returns only the
argmax, so the |xc| vector stored next to it is the reference's own expression (:75-77) evaluated once more.  Inputs
come from the seeded generator ``passiveradar_b200.synth.offset_pair``; nothing from ``oracle/`` or
``passiveradar_b200/csrc`` is involved.  The GPU box has no reference tree; it only reads the .npz files.
"""
from __future__ import annotations

import argparse
import os
import sys
import time

import numpy as np
import scipy.signal as signal

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.environ.get("PR_REFERENCE", "/root/reference"))

from passiveRadar.signal_utils import find_channel_offset, offset_compensation, xcorr   # noqa: E402  (the reference)
from passiveradar_b200 import synth                                                     # noqa: E402

OUT_DIR = os.environ.get("PR_GOLDEN_OUT", HERE)       # tests regenerate into a scratch directory


def save(name, **arrays):
    path = os.path.join(OUT_DIR, name + ".npz")
    np.savez_compressed(path, **arrays)
    print(f"  wrote {name}.npz ({os.path.getsize(path) / 1024:.1f} KiB)")


def offset_case(name, n, planted, kind, nd, nl):
    if kind == "zeros":
        s1 = s2 = np.zeros(n, np.int8)
    else:
        s1, s2 = synth.offset_pair(n, planted, kind)
    t0 = time.perf_counter()
    off = find_channel_offset(s1, s2, nd, nl)
    dt = time.perf_counter() - t0
    B1 = signal.decimate(s1, nd)
    B2 = np.pad(signal.decimate(s2, nd), (nl, nl), 'constant')
    xc = np.abs(signal.correlate(B1, B2, mode='valid'))
    save(name, s1=s1, s2=s2, nd=nd, nl=nl, planted=planted, offset=np.int64(off), xc=xc, seconds=dt)


def offset_main_case(name, n=5_242_880, planted=1234, kind="int8", seed=synth.BASE_SEED + 73, stride=997):
    """main.py:81-83 on the shipped PRconfig.yaml: 10 cpi = 5 242 880 raw int8 entries per channel, nl = 5e6.
    Inputs are regenerated from the seed; stored: offset, top two |xc| values, a strided subsample."""
    s1, s2 = synth.offset_pair(n, planted, kind, seed)
    nd, nl = 1, 5_000_000
    t0 = time.perf_counter()
    off = find_channel_offset(s1, s2, nd, nl)
    dt = time.perf_counter() - t0
    xc = np.abs(signal.correlate(signal.decimate(s1, nd), np.pad(signal.decimate(s2, nd), (nl, nl), 'constant'),
                                 mode='valid'))
    save(name, n=n, planted=planted, kind=kind, seed=seed, nd=nd, nl=nl, offset=np.int64(off),
         top2=np.sort(xc)[-2:][::-1].copy(), stride=stride, xc_sub=xc[::stride].copy(), s1_probe=s1[::100003].copy(),
         seconds=dt)


def xcorr_case(name, n1, n2, nlead, nlag, dtype):
    a, b = synth.offset_pair(max(n1, n2), 37, "complex64", seed=synth.BASE_SEED + 91)
    a, b = a[:n1], b[:n2]
    if np.dtype(dtype).kind == 'c':
        s1, s2 = a.astype(dtype), b.astype(dtype)
    else:
        s1, s2 = a.real.astype(dtype), b.real.astype(dtype)
    out = xcorr(s1, s2, nlead, nlag)
    save(name, s1=s1, s2=s2, nlead=nlead, nlag=nlag, out=out)


def offcomp_case(name, planted):
    x1, x2 = synth.offset_pair(12_000, planted, "complex64", seed=synth.BASE_SEED + 5)
    out = offset_compensation(x1, x2, 8000, 2, 300)
    save(name, x1=x1, x2=x2, ns=8000, ndec=2, nlag=300, out=out, same=np.bool_(out is x2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=None)
    args = ap.parse_args()

    def want(name):
        return args.only is None or args.only in name

    if want("offset_int8_pos"):
        offset_case("offset_int8_pos", 30_000, 173, "int8", nd=1, nl=2000)
    if want("offset_c64_neg"):
        offset_case("offset_c64_neg", 24_000, -411, "complex64", nd=1, nl=1500)
    if want("offset_nd4"):
        offset_case("offset_nd4", 40_000, 96, "int16", nd=4, nl=800)
    if want("offset_zeros"):
        offset_case("offset_zeros", 5_000, 0, "zeros", nd=3, nl=400)
    if want("offset_main"):
        offset_main_case("offset_main")
    for case, n1, n2, nlead, nlag in (("equal", 3000, 3000, 700, 700), ("s2_longer", 1500, 4000, 300, 200),
                                      ("s1_longer", 5000, 1200, 100, 250), ("lead_ne_lag", 2500, 2500, 1200, 90)):
        for dt, tag in ((np.complex64, "c64"), (np.complex128, "c128"), (np.float64, "f64")):
            if want(f"xcorr_{case}_{tag}"):
                xcorr_case(f"xcorr_{case}_{tag}", n1, n2, nlead, nlag, dt)
    if want("offcomp_zero"):
        offcomp_case("offcomp_zero", 0)
    if want("offcomp_shift"):
        offcomp_case("offcomp_shift", -58)


if __name__ == "__main__":
    main()
