"""bench.py's contract, as far as it can be checked without a GPU: BASELINE.json's configuration per GPU
count (the B200 arm and the reference arm print the same `config`), and the reference arm's JSON line
(the reference's own CPU chain, timed on the host cores through oracle/_ref or the C port)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_baseline_configurations_per_gpu_count():
    import bench
    with open(os.path.join(ROOT, "BASELINE.json")) as f:
        base = json.load(f)
    assert "aggregate IQ Msamples/s" in base["metric"] and bench.METRIC == "aggregate_iq_msamples_per_s"
    cfgs = " | ".join(base["configs"])
    assert "1024" in cfgs and "8192" in cfgs and "16384" in cfgs and "65536" in cfgs
    assert bench.BASELINE_CONFIGS[1][:2] == ("am", 1024)          # the headline: AM x1024 on one GPU
    assert bench.BASELINE_CONFIGS[2][:2] == ("ssb", 16384) and bench.BASELINE_CONFIGS[4][:2] == ("ssb", 16384)
    assert bench.BASELINE_CONFIGS[8][:2] == ("mixed", 65536)
    for n, (wl, total, scaling) in bench.BASELINE_CONFIGS.items():
        assert total % n == 0 and scaling in ("weak", "strong")
        assert wl in bench.KERNELS
    cfg = bench.config_of("ssb", "x", "tone", 8192, 2, 2)
    assert cfg["channels_total"] == 16384 and cfg["channels_per_gpu"] == 8192
    assert cfg["iq_bytes_per_gpu_per_step"] == 8192 * 2 * bench.BLOCK_BYTES
    # one step's input must exceed the 126 MB L2 for every workload's default size
    from rtlsdrdiags_b200 import synth
    for wl in ("am", "fm", "wbfm", "ssb", "mixed"):
        ch = synth.WORKLOADS[wl][0]
        assert ch * bench.default_blocks(wl, ch) * bench.BLOCK_BYTES >= 512 << 20


@pytest.mark.parametrize("n_gpus,workload,total", [(1, "am", 1024), (8, "mixed", 65536)])
def test_reference_arm_line(n_gpus, workload, total):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", str(n_gpus),
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "aggregate_iq_msamples_per_s"
    assert line["unit"] == "Msamples/s" and line["higher_is_better"] is True and line["n_gpus"] == n_gpus
    assert line["config"]["workload"] == workload and line["config"]["channels_total"] == total
    assert line["value"] > 0 and line["gpu_launches"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_samples_whole_channels_within_the_budget(tmp_path):
    import numpy as np
    import bench
    pcm = np.repeat(np.arange(-300, 300, dtype=np.int16)[:, None], 1024, axis=1)
    counts = np.arange(600, dtype=np.uint32)
    for d in ("a", "b"):
        (tmp_path / d).mkdir()
        bench.dump_outputs(str(tmp_path / d), pcm, counts, budget=1 << 20)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 1 << 20
    rows = np.load(tmp_path / "a" / "channels.npy")
    got = np.load(tmp_path / "a" / "pcm.npy")
    assert got.dtype == np.float32 and rows.dtype == np.float64 and 0 < rows.size < 600
    assert np.array_equal(got, pcm[rows.astype(np.int64)]) and np.array_equal(np.load(tmp_path / "a" / "counts.npy"), rows)
    for name in ("channels", "pcm", "counts"):  # the sample is fixed
        assert np.array_equal(np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy")))
    (tmp_path / "c").mkdir()
    bench.dump_outputs(str(tmp_path / "c"), pcm[:200], counts[:200], budget=1 << 20)
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "c"), pcm, counts, budget=4096)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(tmp_path / "d")],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "--steps" in r.stderr and not (tmp_path / "d").exists()
    assert sorted(f.name for f in (tmp_path / "c").iterdir()) == ["counts.npy", "pcm.npy"]
    assert np.array_equal(np.load(tmp_path / "c" / "pcm.npy"), pcm[:200])


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(tmp_path):
    """Two runs write the same arrays, and they are the PCM an engine returns after the same number of
    calls on the same input: the untimed warm-up (at least 3) plus the --steps timed ones."""
    import numpy as np
    import torch
    import bench
    import rtlsdrdiags_b200 as R
    from rtlsdrdiags_b200 import synth
    steps, channels, blocks = 4, 40, 2
    nbytes = blocks * bench.BLOCK_BYTES
    args = ["--workload", "mixed", "--channels", str(channels), "--blocks", str(blocks), "--steps", str(steps),
            "--warmup", "1", "--no-extras", "--no-cpu", "--no-e2e"]
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args + ["--dump-outputs", str(tmp_path / d)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
    got = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in ("pcm", "counts")}
    for n, a in got.items():
        assert np.array_equal(a, np.load(tmp_path / "b" / (n + ".npy")))
    modes = synth.modes_for("mixed", channels)
    iq = synth.make_bank("tone", modes, nbytes, 0xB200, torch.device("cuda", 0))
    e = R.Engine(channels, 0, nbytes)
    e.set_modes(modes.numpy())
    for _ in range(3 + steps):
        e.accept_iq_device(iq)
    pcm, counts = e.get_pcm()
    e.close()
    assert got["pcm"].dtype == np.float32 and np.array_equal(got["pcm"], pcm.astype(np.float32))
    assert got["counts"].dtype == np.float64 and np.array_equal(got["counts"], counts)
