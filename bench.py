#!/usr/bin/env python
"""bench.py -- throughput of the IQ->PCM hot path on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload am|fm|wbfm|ssb|mixed]
                    [--signal tone|noise] [--blocks T] [--impl reference] [--no-extras] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic IQ: every channel
of the bank gets T reference blocks (T x 32768 bytes = T x 64 ms of signal) and comes
out as T x 512 PCM samples. Channels shard across ranks with no data-path collective;
torch.distributed is used for the barrier, the max-over-ranks of the device-timed region
and the gather of the per-rank parity flags only.

Without --workload the run is BASELINE.json's configuration for N GPUs:
    N = 1     AM envelope demod, 1024 channels                      (configs[1], the headline)
    N = 2, 4  LSB/USB SSB demod, 16384 channels across the GPUs     (configs[3]; strong scaling 2 -> 4)
    N = 8     mixed AM/FM/WBFM/LSB/USB bank, 65536 channels         (configs[4])
and, for N > 1, a second short run of the headline AM bank per GPU (`am_weak`), so the 1 -> N
weak-scaling curve of the headline exists next to the named configurations.

Prints ONE JSON line (rank 0). `value` is whole-job complex-IQ Msamples/s with the
input already resident in HBM; `e2e` is the same metric through the C ABI with host
buffers (H2D of the IQ and D2H of the PCM inside the timed region); `roofline` puts
the kernel against the measured HBM copy bandwidth; `cpu_baseline` is the reference's
own CPU chain (oracle/_ref) on this box's host cores over a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALGO_BYTES_PER_SAMPLE = 2.0 + 2.0 / 32.0  # 2 B of IQ read + one int16 PCM sample per 32 (SURVEY 8d)
BLOCK_BYTES = 32768
METRIC = "aggregate_iq_msamples_per_s"
# The step is timed as a whole. AM/SSB: the FIR kernel dominates; its small recurrence kernel
# (dc_block_kernel) runs one step behind on a second stream and is inside the timed region.
KERNELS = {"am": "amssb_fir_kernel<false> (+ dc_block_kernel overlapped on the second stream)",
           "ssb": "amssb_fir_kernel<true> (+ dc_block_kernel overlapped on the second stream)",
           "fm": "fm_tile_kernel", "wbfm": "wbfm_tile4_kernel<true> (tcgen05 pre-filter, two channels per worker warp)",
           "mixed": "amssb_fir_kernel<false> + amssb_fir_kernel<true> + 2 x dc_block_kernel + fm_tile_kernel + "
                    "wbfm_tile2_kernel<false> (the step is timed as a whole)"}
# BASELINE.json configs per GPU count: (workload, total channels, scaling label)
BASELINE_CONFIGS = {1: ("am", 1024, "weak"), 2: ("ssb", 16384, "strong"), 4: ("ssb", 16384, "strong"),
                    8: ("mixed", 65536, "weak")}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=0, help="timed steps (0 = enough for ~2 s of device time)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default=None, choices=["am", "fm", "wbfm", "ssb", "mixed"],
                    help="default: BASELINE.json's configuration for --gpus N (see the module docstring)")
    ap.add_argument("--signal", default="tone", choices=["tone", "noise"])
    ap.add_argument("--blocks", type=int, default=0, help="reference blocks per channel per step (0 = auto)")
    ap.add_argument("--channels", type=int, default=0, help="channels per GPU (0 = the workload's)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary per-mode lines")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="tuning runs only: skip the end-to-end leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the PCM and per-channel sample counts of the last timed step "
                         "as DIR/<name>.npy (float32 / float64, at most 64 MB in all: a seeded sample of channels when larger); "
                         "needs --steps K > 0")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the B200 arm computed")
    if args.dump_outputs and args.steps <= 0:
        # the engine's state carries from step to step: comparable dumps need the same number of steps
        ap.error("--dump-outputs needs --steps K > 0")
    return args


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, pcm, counts, suffix="", budget=DUMP_BYTES):
    """The last timed step's results as a caller receives them from sdr_get_pcm: pcm [channels][samples] as float32
    (int16 values, exact) and counts [channels] as float64. Above `budget` bytes a fixed, seeded sample of whole
    channels is written, with their indices in channels.npy, so that two builds can be compared row for row."""
    import numpy as np
    n, samples = pcm.shape
    rows = np.arange(n)
    budget -= 4096  # the three .npy headers
    if n * (samples * 4 + 16) > budget:
        keep = budget // (samples * 4 + 16)
        if keep < 1:
            raise SystemExit("--dump-outputs: one channel's PCM alone exceeds this rank's %d bytes" % budget)
        rows = np.sort(np.random.default_rng(0xD0).choice(n, size=keep, replace=False))
        np.save(os.path.join(out_dir, "channels%s.npy" % suffix), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "pcm%s.npy" % suffix), pcm[rows].astype(np.float32))
    np.save(os.path.join(out_dir, "counts%s.npy" % suffix), counts[rows].astype(np.float64))


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def default_blocks(workload, channels):
    # keep one step's input above the 126 MB L2 (and <= 4 GiB)
    t = 1
    while channels * t * BLOCK_BYTES < 512 * 1024 * 1024:
        t *= 2
    return t


class ClockSampler:
    """nvidia-smi samples DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def _cpu_chain(O, use_ref, modes, iq, cores, want_pcm):
    if use_ref:
        return O.ref_bank(modes, iq, BLOCK_BYTES, cores, want_pcm=want_pcm)
    return O.oracle_bank(modes, iq, BLOCK_BYTES, cores, want_pcm=want_pcm)


def run_cpu_reference(workload, modes_np, n_blocks, seconds_target=6.0, signal="tone", check_gpu=False):
    """The reference's CPU chain on this box's host cores over a bounded sample of the
    workload. Returns (Msamples/s, descriptor dict). Uses oracle/_ref (the unmodified
    reference) when it was built, else the oracle port."""
    import numpy as np
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_binding as O
    from rtlsdrdiags_b200 import synth
    cores = os.cpu_count() or 1
    n_ch = min(int(modes_np.size), 8 * cores)
    modes = np.ascontiguousarray(modes_np[:n_ch])
    t_blocks = min(n_blocks, 4)
    nbytes = t_blocks * BLOCK_BYTES
    iq = synth.make_bank(signal, torch.from_numpy(modes.copy()), nbytes, 1234, "cpu").numpy()
    use_ref = O.ref("radiodiags") is not None
    kind = "reference" if use_ref else "port"
    done, elapsed, reps = 0, 0.0, 0
    while elapsed < seconds_target and reps < 1000:
        _, secs = _cpu_chain(O, use_ref, modes, iq, cores, False)
        elapsed += secs
        done += n_ch * nbytes // 2
        reps += 1
    msps = done / elapsed / 1e6
    desc = {"value": round(msps, 3), "unit": "Msamples/s", "cores": cores, "kind": kind,
            "sample": "%d channels x %d blocks of the %s workload, %d repetitions, %d host threads"
                      % (n_ch, t_blocks, workload, reps, cores)}
    if check_gpu:
        # SURVEY 8(d): the GPU's PCM for this very sample against the PCM the CPU chain just produced
        import rtlsdrdiags_b200 as R
        ref_pcm, _ = _cpu_chain(O, use_ref, modes, iq, cores, True)
        eng = R.Engine(n_ch, 0, BLOCK_BYTES)
        eng.set_modes(modes)
        got, _ = eng.demodulate(iq)  # one reference-sized block per call, state carried
        eng.close()
        desc["gpu_pcm_identical"] = bool(np.array_equal(got, ref_pcm))
    return msps, desc


def capture_baseline(seconds_target=3.0):
    """BASELINE.json's config 1: FM demodulation of a capture through the reference's FmDemodulator
    chain on the CPU (demod.cc:200-323: signed, rotated int8 IQ in 16384-byte reads). The capture it
    names (demodulatorResearch/f135_4.iq) is absent from the reference mount; the stand-in is the
    committed 64 KiB excerpt of demodulatorResearch/yoyo.iq (tests/golden/golden_capture_v1.npz),
    played 32 times in a row (2 MiB, the size of yoyo.iq). One host thread, as demod.cc runs. The GPU
    engine demodulates the same stream and must return the same PCM."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_binding as O
    import rtlsdrdiags_b200 as R
    path = os.path.join(ROOT, "tests", "golden", "golden_capture_v1.npz")
    if not os.path.exists(path):
        return None
    s8 = np.tile(np.load(path)["iq_s8"], 32)
    use_ref = O.ref("research") is not None
    done, elapsed, reps, pcm = 0, 0.0, 0, None
    while elapsed < seconds_target and reps < 200:
        t0 = time.perf_counter()
        if use_ref:
            d = O.RefDemod(O.KIND_FM, "research")
            pcm = d.accept(s8, block=16384)
        else:
            pcm = O.OracleChain(O.VARIANT_RESEARCH).accept_s8(O.MODE_FM, s8)
        elapsed += time.perf_counter() - t0
        done += s8.size // 2
        reps += 1
    eng = R.Engine(1, 0, 16384)
    eng.set_scaling(R.SCALING_RESEARCH)
    eng.set_mode(0, R.MODE_FM)
    got, _ = eng.demodulate(s8.reshape(1, -1), fmt=R.IQ_S8_ROTATED)
    eng.close()
    return {"value": round(done / elapsed / 1e6, 3), "unit": "Msamples/s", "cores": 1,
            "kind": "reference" if use_ref else "port",
            "sample": "FM, 64 KiB excerpt of demodulatorResearch/yoyo.iq x 32 (stand-in for the absent f135_4.iq), "
                      "16384-byte reads, %d repetitions, 1 host thread" % reps,
            "realtime_factor": round(done / elapsed / 256000.0, 1),
            "gpu_pcm_identical": bool(np.array_equal(got[0], pcm))}


def shard_parity(R, synth, workload, channels, first_channel, n_blocks, device_index, signal, seed):
    """This rank's shard against the CPU chain (oracle/_ref, the compiled reference, when it was
    built): a sample of the shard's channels, two passes of the bench's own call shape (n_blocks
    reference blocks per call, so the carried state and the segmented recurrence are exercised as
    timed), PCM compared bit for bit. The CPU chain sees the same bytes in 32768-byte blocks."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_binding as O
    use_ref = O.ref("radiodiags") is not None
    n_s = min(channels, 20)
    pick = np.unique(np.linspace(0, channels - 1, n_s).astype(np.int64))  # spread over the shard
    modes = synth.modes_for(workload, channels, first_channel=first_channel)[pick]
    blocks = min(n_blocks, 4)
    nbytes = blocks * BLOCK_BYTES
    iq = synth.make_bank(signal, modes, 2 * nbytes, seed, "cpu").numpy()
    eng = R.Engine(int(pick.size), device_index, nbytes)
    eng.set_modes(modes.numpy())
    got, _ = eng.demodulate(iq)
    eng.close()
    cores = min(os.cpu_count() or 1, int(pick.size))
    exp, _ = _cpu_chain(O, use_ref, modes.numpy(), iq, cores, True)
    return bool(np.array_equal(got, exp)), {
        "checker": "oracle/_ref (the reference compiled in place)" if use_ref else "oracle port",
        "sample": "%d channels spread over the shard x 2 calls of %d blocks (%s)" % (pick.size, blocks, signal)}


def bench_one(torch, R, synth, workload, channels, n_blocks, steps, warmup, signal, device, rank, world,
              dist, want_e2e=True, first_channel=None, want_outputs=False):
    """Times `steps` passes of one workload on this rank. Returns a dict of local results; with
    want_outputs, res["outputs"] is (pcm, counts) of the last timed step."""
    first = rank * channels if first_channel is None else first_channel
    modes = synth.modes_for(workload, channels, first_channel=first)
    nbytes = n_blocks * BLOCK_BYTES
    eng = R.Engine(channels, device.index, nbytes)
    eng.set_modes(modes.numpy())
    if os.environ.get("SDR_BENCH_TILE_LOADER"):  # A/B runs: AM/SSB tiles by cp.async (0) or TMA with 2..4 buffers
        eng.debug_set_tile_loader(int(os.environ["SDR_BENCH_TILE_LOADER"]))
    if os.environ.get("SDR_BENCH_DC_SHAPE"):     # A/B runs: "segments,warm-up rows" of the recurrence kernel
        eng.debug_set_dc_shape(*[int(x) for x in os.environ["SDR_BENCH_DC_SHAPE"].split(",")])
    # a dedicated (non-default) stream: the kernels are launched on it and the CUDA
    # events that time them are recorded on it
    stream = torch.cuda.Stream(device)
    eng.set_stream(stream.cuda_stream)
    iq = synth.make_bank(signal, modes, nbytes, 0xB200 + rank, device)
    torch.cuda.synchronize(device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def timed(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(n):
            eng.accept_iq_device(iq)
        eng.join()  # the end event must cover the engine's second stream too
        b.record(stream)
        return a, b

    # ---- device-resident: the kernel(s) alone ----
    a, b = timed(max(warmup, 3))  # untimed warm-up: includes the engine's lazy allocations
    barrier()
    if steps <= 0:  # auto: about two seconds of device time, identical on every rank
        a, b = timed(20)          # calibration on the warmed-up engine
        barrier()
        per = reduce_max(torch, dist, world, device, a.elapsed_time(b) / 20)
        steps = int(min(20000, max(30, 2000.0 / max(per, 1e-3))))
    l0 = eng.launch_count
    sampler = ClockSampler(device.index) if rank == 0 and not os.environ.get("SDR_BENCH_NO_SAMPLER") else None
    barrier()
    e0, e1 = timed(steps)
    barrier()
    clocks = sampler.stop() if sampler else None
    # read back before the clock soak below runs further steps on the same engine
    outputs = eng.get_pcm() if want_outputs else None
    ms = e0.elapsed_time(e1)
    launches = eng.launch_count - l0
    redo = eng.debug_dc_redo_count()
    if clocks is not None:
        clocks["sampled"] = "timed region"
        if clocks["samples"] < 5:  # region too short for nvidia-smi: soak the same call for 1.5 s
            sampler = ClockSampler(device.index)
            t_end = time.time() + 1.5
            while time.time() < t_end:
                timed(20)
                torch.cuda.synchronize(device)
            clocks = sampler.stop()
            clocks["sampled"] = "1.5 s soak of the same launch right after the timed region (region too short)"
    res = {"ms_total": ms, "launches": launches, "clocks": clocks, "steps": steps,
           "samples_per_step": channels * nbytes // 2, "h2d": channels * nbytes,
           "d2h": channels * (nbytes // 64) * 2, "dc_redo": redo, "outputs": outputs}
    eng.set_stream(0)
    eng.close()

    # ---- end to end through the C ABI: pinned host IQ in, host PCM out, every step ----
    if want_e2e:
        h_iq = torch.empty((channels, nbytes), dtype=torch.uint8, pin_memory=True)
        h_iq.copy_(iq)
        del iq
        h_pcm = torch.empty((channels, nbytes // 64), dtype=torch.int16, pin_memory=True)
        torch.cuda.synchronize(device)
        n_warm, n_e2e = 3, 10
        # Both paths start from a fresh engine and see the same 13 ticks, so their last PCM must agree.
        # (1) one synchronous call pair per step: sdr_accept_iq(host) + sdr_get_pcm
        eng = R.Engine(channels, device.index, nbytes)
        eng.set_modes(modes.numpy())
        for _ in range(n_warm):
            eng.accept_iq_ptr(h_iq.data_ptr(), nbytes, nbytes, R.IQ_HOST)
            eng.get_pcm_ptr(h_pcm.data_ptr())
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            eng.accept_iq_ptr(h_iq.data_ptr(), nbytes, nbytes, R.IQ_HOST)
            eng.get_pcm_ptr(h_pcm.data_ptr())  # synchronises: the step's result is on the host
        torch.cuda.synchronize(device)
        res["e2e_sync_ms_total"] = (time.perf_counter() - t0) * 1e3
        sync_sum = int(h_pcm.to(torch.int64).sum().item())
        del h_pcm
        eng.close()
        # (2) the ingest ring (the bank's DataConsumer): every step's tick is taken from a pinned
        # slot, copied to the GPU, demodulated and its PCM copied back to pinned memory; copies
        # of neighbouring ticks overlap. A step is complete when its tick has been retired. The
        # producer writes in place: sdr_ingest_acquire hands it the pinned slot, so no host copy
        # is part of a step (sdr_ingest_accept, which copies like DataConsumer.cc:246-248, is
        # timed separately below).
        eng = R.Engine(channels, device.index, nbytes)
        eng.set_modes(modes.numpy())
        ring = R.Ingest(eng, 3, nbytes)
        for _ in range(n_warm):                # fill the three pinned slots with the workload
            ring.acquire()[:] = h_iq.numpy()
            ring.commit(0)
        for _ in range(n_warm):
            ring.retire(copy=False)
        barrier()
        t0 = time.perf_counter()
        acc = 0
        for k in range(n_e2e):
            ring.commit(k)                    # the slot's content is this step's input
            if k >= 2:
                _, pcm, _ = ring.retire(copy=False)
                acc += int(pcm[0, 0])
        for _ in range(min(2, n_e2e)):
            _, pcm, _ = ring.retire(copy=False)
            acc += int(pcm[0, 0])
        torch.cuda.synchronize(device)
        res["e2e_ms_total"] = (time.perf_counter() - t0) * 1e3
        res["e2e_steps"] = n_e2e
        ring_sum = int(torch.from_numpy(pcm.copy()).to(torch.int64).sum().item())
        res["pcm_checksum"] = ring_sum
        res["e2e_paths_agree"] = ring_sum == sync_sum
        # (3) the copying entry: sdr_ingest_accept memcpy's the caller's block into the slot first
        n_copy = 3
        barrier()
        t0 = time.perf_counter()
        for k in range(n_copy):
            ring.accept(k, h_iq.numpy())
            if k >= 2:
                ring.retire(copy=False)
        for _ in range(min(2, n_copy)):
            ring.retire(copy=False)
        torch.cuda.synchronize(device)
        res["e2e_copy_ms_total"] = (time.perf_counter() - t0) * 1e3
        res["e2e_copy_steps"] = n_copy
        ring.close()
        eng.close()
        del h_iq
    else:
        del iq
    torch.cuda.empty_cache()
    return res


def reduce_max(torch, dist, world, device, x):
    if world == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def gather_flags(torch, dist, world, device, flag):
    if world == 1:
        return [bool(flag)]
    t = torch.tensor([1 if flag else 0], dtype=torch.int32, device=device)
    out = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return [bool(int(x.item())) for x in out]


def traffic_for(workload):
    """DRAM bytes per launch of the workload's dominant kernel from this round's ncu --set full
    capture (profiles/ncu_traffic.json), with the label of the build it was captured on."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            d = json.load(f)
        return d.get(workload), d.get("_captured")
    except Exception:
        return None, None


def config_of(workload, wl_desc, signal, channels, world, n_blocks):
    """The `config` object of the JSON line: identical for the B200 arm and the reference arm."""
    per_gpu = channels * n_blocks * BLOCK_BYTES
    return {"workload": workload, "description": wl_desc, "signal": signal,
            "channels_per_gpu": channels, "channels_total": channels * world,
            "blocks_per_channel_per_step": n_blocks,
            "block_bytes": BLOCK_BYTES, "iq_bytes_per_gpu_per_step": per_gpu,
            "l2": "input per step (%d MiB) exceeds the 126 MB L2; no flush needed" % (per_gpu >> 20),
            "sharding": "contiguous channel ranges per rank, no data-path collective"}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    import numpy as np
    from rtlsdrdiags_b200 import synth
    n_gpus = world if args.impl != "reference" else max(args.gpus, 1)
    scaling = "weak"
    total_channels = None
    if args.workload is None:
        workload, total_channels, scaling = BASELINE_CONFIGS.get(n_gpus, ("am", 1024 * n_gpus, "weak"))
        channels = args.channels or total_channels // n_gpus
        if n_gpus == 1:
            total_channels = None
    else:
        workload = args.workload
        channels = args.channels or synth.WORKLOADS[workload][0]
    wl_desc = synth.WORKLOADS[workload][2] if total_channels is None else \
        "%s (%d channels in total, %d per GPU on %d GPUs)" % (synth.WORKLOADS[workload][2], total_channels,
                                                               channels, n_gpus)
    n_blocks = args.blocks or default_blocks(workload, channels)

    if args.impl == "reference":
        # the reference's own CPU implementation of the path, all host threads; rank 0 only
        if rank != 0:
            return 0
        modes = synth.modes_for(workload, channels).numpy()
        vals = []
        desc = None
        n_steps = args.steps if args.steps > 0 else 5
        for i in range(args.warmup + n_steps):
            v, desc = run_cpu_reference(workload, modes, n_blocks, seconds_target=1.0, signal=args.signal)
            if i >= args.warmup:
                vals.append(v)
        value = float(np.mean(vals)) if vals else v
        desc["value"] = round(value, 3)
        line = {"impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": "Msamples/s",
                "n_gpus": args.gpus, "steps": len(vals), "warmup": args.warmup,
                "ms_per_step": None, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
                "dtype": "q15 int32 + f32", "data": "synthetic",
                "config": config_of(workload, wl_desc, args.signal, channels, n_gpus, n_blocks),
                "note": "each step times a bounded sample of this workload on the host cores (see "
                        "cpu_baseline.sample); the CPU arm does not scale with --gpus",
                "realtime_channels": round(value / 0.256, 1), "cpu_baseline": desc,
                "e2e": {"value": round(value, 3), "unit": "Msamples/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    import torch
    import rtlsdrdiags_b200 as R
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path")
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    if world != args.gpus and rank == 0:
        print("note: --gpus %d but WORLD_SIZE %d; using WORLD_SIZE" % (args.gpus, world), file=sys.stderr)

    res = bench_one(torch, R, synth, workload, channels, n_blocks, args.steps, args.warmup, args.signal,
                    device, rank, world, dist, want_e2e=not args.no_e2e, want_outputs=bool(args.dump_outputs))
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        dump_outputs(args.dump_outputs, *res.pop("outputs"), suffix="_rank%d" % rank if world > 1 else "",
                     budget=DUMP_BYTES // world)  # DUMP_BYTES for the whole job
    if args.no_e2e:
        res.update(e2e_ms_total=float("inf"), e2e_sync_ms_total=float("inf"), e2e_copy_ms_total=float("inf"),
                   e2e_steps=0, e2e_copy_steps=0, e2e_paths_agree=None)
    ms_total = reduce_max(torch, dist, world, device, res["ms_total"])
    e2e_ms_total = reduce_max(torch, dist, world, device, res["e2e_ms_total"])
    total_samples_step = res["samples_per_step"] * world
    steps = res["steps"]
    value = total_samples_step * steps / (ms_total * 1e-3) / 1e6
    e2e_value = total_samples_step * res["e2e_steps"] / (e2e_ms_total * 1e-3) / 1e6
    e2e_sync_ms = reduce_max(torch, dist, world, device, res["e2e_sync_ms_total"])
    e2e_sync_value = total_samples_step * res["e2e_steps"] / (e2e_sync_ms * 1e-3) / 1e6
    e2e_copy_ms = reduce_max(torch, dist, world, device, res["e2e_copy_ms_total"])
    e2e_copy_value = total_samples_step * res["e2e_copy_steps"] / (e2e_copy_ms * 1e-3) / 1e6
    paths_agree = gather_flags(torch, dist, world, device, bool(res["e2e_paths_agree"]))
    peak, peak_src = peaks()
    # the dominant kernel: one launch per demodulator kind per step; for single-mode
    # workloads that is the only kernel in the timed region besides the small recurrence kernel
    kernel_ms = res["ms_total"] / steps
    achieved = res["samples_per_step"] * ALGO_BYTES_PER_SAMPLE / (kernel_ms * 1e-3) / 1e9
    traffic, traffic_label = traffic_for(workload)

    # every rank: a sample of ITS shard against the compiled reference
    ok, parity_desc = shard_parity(R, synth, workload, channels, rank * channels, n_blocks, device.index,
                                   args.signal, 4321 + rank)
    per_rank = gather_flags(torch, dist, world, device, ok)

    # N > 1: the headline AM bank per GPU as well, so its weak-scaling curve exists
    am_weak = None
    if world > 1 and workload != "am" and not args.no_extras:
        ch = synth.WORKLOADS["am"][0]
        nb = default_blocks("am", ch)
        r = bench_one(torch, R, synth, "am", ch, nb, 200, 5, args.signal, device, rank, world, dist, want_e2e=False)
        ms_am = reduce_max(torch, dist, world, device, r["ms_total"])
        v = r["samples_per_step"] * world * r["steps"] / (ms_am * 1e-3) / 1e6
        am_weak = {"value": round(v, 1), "unit": "Msamples/s", "channels_per_gpu": ch, "blocks": nb, "steps": r["steps"],
                   "ms_per_step": round(ms_am / r["steps"], 4), "scaling": "weak",
                   "roofline_frac": round(v * 1e6 * ALGO_BYTES_PER_SAMPLE / 1e9 / (peak * world), 4)}

    extras = {}
    if rank == 0 and world == 1 and not args.no_extras:
        for wl in ["fm", "wbfm", "ssb", "mixed", "am"]:
            if wl == workload:
                continue
            ch = synth.WORKLOADS[wl][0]
            nb = default_blocks(wl, ch)
            r = bench_one(torch, R, synth, wl, ch, nb, 40, 3, args.signal, device, 0, 1, None, want_e2e=False)
            v = r["samples_per_step"] * r["steps"] / (r["ms_total"] * 1e-3) / 1e6
            extras[wl] = {"value": round(v, 1), "unit": "Msamples/s", "channels": ch, "blocks": nb,
                          "realtime_channels": round(v / 0.256),
                          "roofline_frac": round(v * 1e6 * ALGO_BYTES_PER_SAMPLE / 1e9 / peak, 4)}
            if not args.no_cpu:  # the reference's CPU chain on the same workload, bounded sample
                _, c = run_cpu_reference(wl, synth.modes_for(wl, ch).numpy(), nb, seconds_target=2.0,
                                         signal=args.signal, check_gpu=True)
                extras[wl]["cpu_baseline"] = c
        if args.signal == "tone":
            r = bench_one(torch, R, synth, workload, channels, n_blocks, 40, 3, "noise", device, 0, 1,
                          None, want_e2e=False)
            v = r["samples_per_step"] * r["steps"] / (r["ms_total"] * 1e-3) / 1e6
            extras[workload + "_noise_input"] = {"value": round(v, 1), "unit": "Msamples/s"}

    cpu = None
    if rank == 0 and not args.no_cpu:
        modes = synth.modes_for(workload, channels).numpy()
        _, cpu = run_cpu_reference(workload, modes, n_blocks, seconds_target=12.0 if world == 1 else 4.0,
                                   signal=args.signal, check_gpu=True)

    config1 = capture_baseline() if rank == 0 and world == 1 and not args.no_cpu else None

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": "Msamples/s",
            "n_gpus": world, "steps": steps, "warmup": max(args.warmup, 3),
            "ms_per_step": round(ms_total / steps, 4), "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "q15 int32 + f32", "data": "synthetic",
            "config": config_of(workload, wl_desc, args.signal, channels, world, n_blocks),
            "realtime_channels": round(value / 0.256),
            "realtime_channels_per_gpu": round(value / 0.256 / world),
            "clocks": res["clocks"],
            "e2e": {"value": round(e2e_value, 2), "unit": "Msamples/s", "h2d_bytes_per_step": res["h2d"] * world,
                    "d2h_bytes_per_step": res["d2h"] * world, "steps": res["e2e_steps"],
                    "api": "sdr_ingest_acquire/commit + sdr_ingest_retire: 3-slot pinned ring the producer writes "
                           "in place, every tick copied host->device, demodulated, PCM copied device->host; "
                           "neighbouring ticks overlap",
                    "synchronous_value": round(e2e_sync_value, 2),
                    "synchronous_api": "sdr_accept_iq(SDR_IQ_HOST) + sdr_get_pcm per step, pinned host buffers",
                    "copying_value": round(e2e_copy_value, 2),
                    "copying_api": "sdr_ingest_accept: the caller's block is first memcpy'd into the pinned slot "
                                   "by one host thread (DataConsumer.cc:246-248), then as above",
                    "paths_agree": all(paths_agree)},
            "gpu_launches": res["launches"],
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_capture": traffic_label,
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_sample": ALGO_BYTES_PER_SAMPLE,
                         "kernel_ms": round(kernel_ms, 4), "kernel": KERNELS[workload],
                         "frac_of_box": round(value * 1e6 * ALGO_BYTES_PER_SAMPLE / 1e9 / (peak * world), 4)},
            "parity": {"gpu_pcm_identical": all(per_rank), "per_rank": per_rank, **parity_desc,
                       "recurrence_segments_redone_in_timed_region": res["dc_redo"]},
            "cpu_baseline": cpu,
            "cpu_baseline_config1_capture": config1,
            "am_weak": am_weak,
            "other_workloads": extras,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
