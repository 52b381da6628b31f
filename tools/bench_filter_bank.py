#!/usr/bin/env python
"""Throughput of the batched filter banks on one GPU (device-resident rows larger than L2,
CUDA events on the bank's stream). One JSON line per case: input samples/s, algorithmic GB/s
(bytes read + bytes written) and the fraction of the measured HBM peak. The first line names the
card and its power limit, read in the same run."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rtlsdrdiags_b200 as R  # noqa: E402


def lowpass(n_taps, cutoff, gain=1.0):
    k = np.arange(n_taps) - (n_taps - 1) / 2.0
    h = 2 * cutoff * np.sinc(2 * cutoff * k) * np.hamming(n_taps)
    return (gain * h / h.sum()).astype(np.float32)


def peak_gbs():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        return 6553.6


CASES = [  # name, kind, taps, factor, rows, samples per row
    ("decimator_f32 80 taps 4:1 (decimateAudio.cc shape)", R.FILTER_DECIMATOR_F32, lowpass(80, 0.11), 4, 4096, 65536),
    ("decimator_i16 80 taps 4:1 (Int16/decimateAudio.cc shape)", R.FILTER_DECIMATOR_I16, lowpass(80, 0.11), 4, 4096, 131072),
    ("decimator_i16 8 taps 4:1 (AM stage 1 shape)", R.FILTER_DECIMATOR_I16, lowpass(8, 0.1), 4, 4096, 131072),
    ("interpolator_f32 64 taps 1:2 (interpolateAudio.cc shape)", R.FILTER_INTERPOLATOR_F32, lowpass(64, 0.22, 2.0), 2, 4096, 32768),
    ("interpolator_i16 64 taps 1:2", R.FILTER_INTERPOLATOR_I16, lowpass(64, 0.22, 1.99), 2, 4096, 65536),
    ("fir_f32 7 taps 1:1 (FirFilter shape)", R.FILTER_DECIMATOR_F32, lowpass(7, 0.2), 1, 4096, 32768),
]


STABLE_4 = (np.array([0.05, 0.1, 0.2, 0.1, 0.05], dtype=np.float32),   # nb = 5
            np.poly([0.8, -0.7, 0.6 + 0.3j, 0.6 - 0.3j]).real.astype(np.float32)[[4, 1, 2, 3]])  # na = 4, poles < 0.9
IIR_CASES = [  # name, b, a, rows, samples per row, forced segments per row (0 = automatic)
    ("(a) iir WBFM de-emphasis", [0.0253863, 0.0253863], [-0.9492274], 4096, 65536, 0),
    ("(b) iir DC block", [1, -1], [-0.95], 65535, 8192, 0),   # the most rows a bank takes
    ("(c) iir de-emphasis, 64 long rows", [0.0253863, 0.0253863], [-0.9492274], 64, 16 << 20, 0),
    ("(d) iir stable nb=5 na=4", STABLE_4[0], STABLE_4[1], 4096, 65536, 0),
    ("(e) iir de-emphasis, 64 long rows, one segment per row", [0.0253863, 0.0253863], [-0.9492274], 64, 16 << 20, 1),
]


def card():
    import subprocess
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi unavailable: %s" % e
    return {"card": torch.cuda.get_device_name(0), "nvidia_smi": q}


def bench_iir(peak, stream):
    for name, b, a, rows, n, seg in IIR_CASES:
        x = (torch.rand((rows, n), device="cuda") * 20000 - 10000).contiguous()
        y = torch.zeros((rows, n), device="cuda")
        torch.cuda.synchronize()   # x is written on torch's stream, read on the bank's
        bank = R.IirFilterBank(rows, b, a)
        if seg:
            bank.debug_set_iir_shape(seg)
        bank.set_stream(stream.cuda_stream)
        steps = 3 if seg == 1 else 10   # the serial case takes seconds a call
        with torch.cuda.stream(stream):
            for _ in range(2):
                bank.run_device(x.data_ptr(), n, n, y.data_ptr(), n)
        redo0 = bank.debug_redo_count()
        with torch.cuda.stream(stream):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps):
                bank.run_device(x.data_ptr(), n, n, y.data_ptr(), n)
            e1.record(stream)
        e1.synchronize()
        ms = e0.elapsed_time(e1) / steps
        gbs = rows * n * 8 / (ms * 1e-3) / 1e9   # float in + float out
        print(json.dumps({"case": name, "rows": rows, "samples_per_row": n, "ms": round(ms, 4),
                          "input_msamples_per_s": round(rows * n / ms / 1e3, 1),
                          "algorithmic_gbs": round(gbs, 1), "hbm_peak_gbs": peak, "frac": round(gbs / peak, 4),
                          "nb": len(b), "na": len(a),
                          "segments_redone_per_call": round((bank.debug_redo_count() - redo0) / steps, 1)}))
        bank.close()
        del x, y


def main():
    peak = peak_gbs()
    stream = torch.cuda.Stream()
    print(json.dumps(card()))
    if "--iir" in sys.argv:
        bench_iir(peak, stream)
        return
    for name, kind, taps, factor, rows, n in CASES:
        f32 = kind in (R.FILTER_DECIMATOR_F32, R.FILTER_INTERPOLATOR_F32)
        interp = kind in (R.FILTER_INTERPOLATOR_F32, R.FILTER_INTERPOLATOR_I16)
        dt = torch.float32 if f32 else torch.int16
        x = (torch.rand((rows, n), device="cuda") * 20000 - 10000).round().to(dt).contiguous()
        n_out = n * factor if interp else n // factor
        y = torch.zeros((rows, n_out), device="cuda", dtype=dt)
        b = R.FilterBank(kind, rows, taps, factor)
        b.set_stream(stream.cuda_stream)
        with torch.cuda.stream(stream):
            for _ in range(3):
                b.run_device(x.data_ptr(), n, n, y.data_ptr(), n_out)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            steps = 10
            e0.record(stream)
            for _ in range(steps):
                b.run_device(x.data_ptr(), n, n, y.data_ptr(), n_out)
            e1.record(stream)
        e1.synchronize()
        ms = e0.elapsed_time(e1) / steps
        esize = 4 if f32 else 2
        gbs = (rows * n + rows * n_out) * esize / (ms * 1e-3) / 1e9
        print(json.dumps({"case": name, "rows": rows, "samples_per_row": n, "ms": round(ms, 4),
                          "input_msamples_per_s": round(rows * n / ms / 1e3, 1),
                          "algorithmic_gbs": round(gbs, 1), "hbm_peak_gbs": peak, "frac": round(gbs / peak, 4),
                          "mac_per_input_sample": taps.size / factor if not interp else taps.size}))
        b.close()
    bench_iir(peak, stream)


if __name__ == "__main__":
    main()
