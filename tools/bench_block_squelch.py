#!/usr/bin/env python
"""What gating every 32768-byte block of a multi-block call costs (sdr_set_squelch_block_bytes).

    python tools/bench_block_squelch.py [--steps K] [--warmup W] [--rounds R] [--out FILE.jsonl]

Two banks, AM x1024 and mixed x8192, fed 16-block calls (16 x 32768 bytes per channel, one second of
signal) from device memory; one call's input (512 MiB, 4 GiB) is larger than the B200's L2. The stream
repeats loud, quiet, quiet, quiet blocks; every radio's squelch is armed between the two levels, so with
the one-block tail half of the blocks are open. Three variants, alternated round by round in one run:

  per_call   the squelch block at 0: one decision per 16-block call (every call open)
  per_block  the squelch block at 32768: a decision, and a demodulation pass, per block
  calls_32k  the same stream as sixteen 32768-byte calls with the squelch block at 0 (the workaround
             per_block replaces; same gates and PCM)

A step is one 16-block call (16 calls for calls_32k), timed by the host clock over K steps that end in
a device synchronise. Writes one JSON line per (bank, variant, round) after a line with the card's
name and power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BLOCK = 32768
BLOCKS = 16
PATTERN = [40.0, 1.0, 1.0, 1.0]  # per-block noise amplitude: the loud block, its tail, two closed blocks
THRESHOLD = -12                  # dBFS: between the two levels


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi unavailable: %s" % e
    return q


def make_input(torch, n):
    g = torch.Generator(device="cuda")
    g.manual_seed(0xB10C)
    iq = torch.empty((n, BLOCKS * BLOCK), dtype=torch.uint8, device="cuda")
    for k in range(BLOCKS):
        x = torch.randn((n, BLOCK), generator=g, device="cuda") * PATTERN[k % len(PATTERN)] + 128.0
        iq[:, k * BLOCK:(k + 1) * BLOCK] = x.round_().clamp_(0, 255).to(torch.uint8)
        del x
    return iq


def engine(R, n, modes, setting):
    e = R.Engine(n, 0, BLOCKS * BLOCK)
    e.set_modes(modes)
    for ch in range(n):
        e.set_squelch_threshold(ch, THRESHOLD)
    e.set_squelch_block_bytes(setting)
    return e


def step(e, iq, variant):
    if variant == "calls_32k":
        for k in range(BLOCKS):
            e.accept_iq_device(iq[:, k * BLOCK:(k + 1) * BLOCK])
    else:
        e.accept_iq_device(iq)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    import rtlsdrdiags_b200 as R
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement runs on the GPU only")
    lines = [{"tool": "bench_block_squelch", "card": card(), "torch_device": torch.cuda.get_device_name(0),
              "block_bytes": BLOCK, "blocks_per_call": BLOCKS, "pattern": PATTERN, "threshold_dbfs": THRESHOLD}]
    print(json.dumps(lines[0]), flush=True)
    variants = {"per_call": 0, "per_block": BLOCK, "calls_32k": 0}
    for bank, n in (("am", 1024), ("mixed", 8192)):
        modes = np.full(n, R.MODE_AM, dtype=np.uint8) if bank == "am" else \
            np.array([1 + ch % 5 for ch in range(n)], dtype=np.uint8)
        iq = make_input(torch, n)
        torch.cuda.synchronize()
        engines = {v: engine(R, n, modes, s) for v, s in variants.items()}
        info = {}
        for v, e in engines.items():
            for _ in range(a.warmup):
                step(e, iq, v)
            e.sync()
            before = e.launch_count
            step(e, iq, v)
            _, counts = e.get_pcm()
            allowed, _ = e.get_signal_blocks()
            info[v] = {"launches_per_step": e.launch_count - before, "open_fraction_of_last_call": float(allowed.mean()),
                       "pcm_samples_last_call": int(counts.sum())}
        for r in range(a.rounds):
            for v, e in engines.items():
                e.sync()
                t0 = time.perf_counter()
                for _ in range(a.steps):
                    step(e, iq, v)
                e.sync()
                dt = (time.perf_counter() - t0) / a.steps
                msps = n * BLOCKS * BLOCK / 2 / dt / 1e6
                line = {"bank": bank, "channels": n, "variant": v, "round": r, "steps": a.steps,
                        "ms_per_16_blocks": round(dt * 1e3, 4), "iq_msamples_per_s": round(msps, 1), **info[v]}
                print(json.dumps(line), flush=True)
                lines.append(line)
        for e in engines.values():
            e.close()
        del iq
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
