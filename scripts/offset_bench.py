#!/usr/bin/env python
"""Time find_channel_offset at the shapes main.py runs it (main.py:54, :83), next to the reference's own function.

    python scripts/offset_bench.py [--reps 20] [--out profiles/offset_bench.json] [--no-ref]

Per shape: the device-resident prc_channel_offset (CUDA events around `reps` calls after warm-up, inputs already in
HBM), the host-array drop-in end to end (upload included), and the reference's find_channel_offset on the same box
(baseline/_ref when present, else the oracle's restatement; CPU).  The traffic model beside the time counts the
transform passes at P points of 8 bytes (two column + two row passes forward, the product row pass reads two
planes and writes one, the last column pass reads one).  Appends one JSON line per run to --out.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SHAPES = [("int8", 5242880, 1234, "main.py:83, shipped PRconfig.yaml (10 cpi of int8 entries)"),
          ("complex64", 2621440, -2345, "main.py:54, interleaved input (20 cpi deinterleaved, every 2nd sample)"),
          ("int8", 10485760, 777, "main.py:83 with cpi_seconds_nominal: 4 (tiled: 2 x 2 transforms)")]
COPY_BW = 6.57e12          # bytes/s, DESIGN.md section 4 (measured device-to-device copy)


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:
        power = None
    return name, power


def reference_fn():
    ref = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(os.path.join(ref, "passiveRadar")):
        sys.path.insert(0, ref)
        from passiveRadar.signal_utils import find_channel_offset
        return find_channel_offset, "reference"
    from oracle.offset_oracle import channel_offset_oracle
    return (lambda a, b, nd, nl: channel_offset_oracle(a, b, nd, nl)[0]), "oracle"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "offset_bench.json"))
    ap.add_argument("--no-ref", action="store_true")
    args = ap.parse_args()

    import torch
    import passiveradar_b200 as prb
    from passiveradar_b200 import _lib, synth
    from passiveradar_b200.signal_utils import _decimate_sos, _xcorr_window

    name, power = gpu_info()
    dev = 0
    stream = torch.cuda.Stream(dev)              # a real stream: the legacy default stream would be NULL to the library
    lib = _lib.load()
    ref_fn, ref_kind = reference_fn()
    nd, nl = 1, 5000000
    rows = []
    for kind, n, planted, what in SHAPES:
        s1, s2 = synth.offset_pair(n, planted, kind)
        sig = {"int8": _lib.SIG_I8, "complex64": _lib.SIG_C64}[kind]
        sos, _ = _decimate_sos(nd, kind == "complex64")
        t1, t2 = torch.from_numpy(s1).cuda(dev), torch.from_numpy(s2).cuda(dev)
        doff = torch.zeros(1, dtype=torch.int64, device="cuda:0")
        torch.cuda.synchronize()

        def call():
            _lib.check(lib.prc_channel_offset(t1.data_ptr(), n, t2.data_ptr(), n, sig, nd, nl, sos.ctypes.data,
                                              sos.shape[0], doff.data_ptr(), None, _lib.MEM_DEVICE, dev,
                                              C.c_void_p(stream.cuda_stream), _lib.FLAG_ASYNC))
        for _ in range(args.warmup):
            call()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(args.reps):
            call()
        b.record(stream)
        torch.cuda.synchronize()
        dev_ms = a.elapsed_time(b) / args.reps
        assert int(doff.item()) == planted
        doff.zero_()
        call()
        torch.cuda.synchronize()
        assert int(doff.item()) == planted
        host = []
        for _ in range(3):
            t0 = time.perf_counter()
            off = prb.find_channel_offset(s1, s2, nd, nl)
            host.append(time.perf_counter() - t0)
        assert off == planted
        ref_s = None
        if not args.no_ref:
            t0 = time.perf_counter()
            ref_off = ref_fn(s1, s2, nd, nl)
            ref_s = time.perf_counter() - t0
            assert ref_off == planted
        lag0, nlags = _xcorr_window(n, n, nl, nl)
        need = n + nlags - 1
        P, ntr = (1 << 24), 1
        if need <= 1 << 24:
            P = 1 << 20
            while P < need:
                P <<= 1
        else:
            ntr = 4                                           # 2 lag tiles x 2 x-segments
        traffic = 7 * P * 8 * ntr
        row = {"shape": f"{kind} x {n}", "what": what, "P": P, "transforms": ntr, "device_ms": round(dev_ms, 4),
               "host_call_s": round(min(host), 4), "reference_s": None if ref_s is None else round(ref_s, 3),
               "reference_kind": ref_kind, "traffic_GB": round(traffic / 1e9, 3),
               "traffic_floor_ms": round(traffic / COPY_BW * 1e3, 3)}
        rows.append(row)
        print(json.dumps(row))
        del t1, t2
    rec = {"gpu": name, "power_limit_W": power, "reps": args.reps, "nd": nd, "nl": nl, "rows": rows,
           "time": time.strftime("%Y-%m-%dT%H:%M:%S")}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        f.write(json.dumps(rec) + "\n")
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
