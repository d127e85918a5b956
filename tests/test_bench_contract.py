"""bench.py prints exactly one JSON line with the keys the driver reads."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def run(cmd, timeout=600):
    p = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    return lines


def test_reference_arm_prints_one_json_line():
    lines = run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0",
                 "--log2-frames", "16"])
    assert len(lines) == 1
    b = json.loads(lines[0])
    assert BASE_KEYS <= set(b)
    assert b["impl"] == "reference" and b["unit"] == "Msamples/s" and b["value"] > 0 and b["gpu_launches"] == 0
    assert b["cpu_baseline"]["kind"] in ("reference", "port") and b["cpu_baseline"]["cores"] >= 1
    assert b["e2e"] == {"value": b["value"], "unit": b["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in b["config"] and "model" not in b["config"]


def test_reference_arm_under_torchrun_only_rank0_prints():
    lines = run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                 "--master-addr", "127.0.0.1", "--master-port", "29533", "bench.py", "--gpus", "2",
                 "--impl", "reference", "--steps", "1", "--warmup", "0", "--log2-frames", "16"])
    payload = [l for l in lines if l.startswith("{")]
    assert len(payload) == 1 and json.loads(payload[0])["n_gpus"] == 2


@pytest.mark.gpu
def test_gpu_arm_prints_one_json_line_with_roofline_and_e2e():
    lines = run([sys.executable, "bench.py", "--steps", "4", "--warmup", "3", "--log2-frames", "22",
                 "--e2e-log2-frames", "20", "--cpu-log2-frames", "18", "--min-seconds", "0.2"])
    assert len(lines) == 1
    b = json.loads(lines[0])
    assert BASE_KEYS | {"roofline", "clocks"} <= set(b)
    assert b["gpu_launches"] == 8 and b["n_gpus"] == 1 and b["scaling"] == "weak" and b["vs_baseline"] is None
    r = b["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    e = b["e2e"]
    assert e["h2d_bytes_per_step"] == 2 * 8 * (1 << 20) == e["d2h_bytes_per_step"]
    assert e["value"] > 0 and e["value"] != b["value"] and e["gpu_launches"] > 0
    assert "readStream" in e["api"] and e["raw_link_gbs_per_rank"]["both_each_way_gbs"][0] > 0
    assert e["plugin_rows"] and {"product_pageable_us", "product_pin1_us", "product_library_pinned_us"} <= set(e["plugin_rows"][0])
    assert b["sustained"]["seconds"] >= 0.2
    assert b["cpu_baseline"]["kind"] in ("reference", "port")
    assert isinstance(b["clocks"]["reasons"], list)


@pytest.mark.gpu
@pytest.mark.parametrize("log2_frames", [16, 22], ids=["whole_block", "sampled_block"])
def test_gpu_arm_dumps_what_the_last_timed_step_computed(oracle, tmp_path, log2_frames):
    import numpy as np
    import bench
    import sxtest
    frames = 1 << log2_frames
    lines = run([sys.executable, "bench.py", "--steps", "2", "--warmup", "1", "--log2-frames", str(log2_frames),
                 "--e2e-log2-frames", "16", "--min-seconds", "0", "--no-rows", "--no-cpu-baseline",
                 "--dump-outputs", str(tmp_path)])
    assert len(lines) == 1
    b = json.loads(lines[0])
    assert b["steps"] == 2 and b["gpu_launches"] == 2 * 2     # one RX and one TX launch per timed step
    cf, words = np.load(tmp_path / "rx_cf32.npy"), np.load(tmp_path / "tx_i2s.npy")
    assert cf.dtype == np.float32 and words.dtype == np.float64
    want_cf = sxtest.oracle_rx(oracle, sxtest.synth_frames(oracle, 0, frames, bench.SEED))
    want_words = sxtest.oracle_tx(oracle, want_cf, bench.THR2)
    pick = bench.dump_frames(frames)
    if pick is not None:
        assert pick.size == bench.DUMP_FRAMES and np.array_equal(pick, bench.dump_frames(frames))
        keep = np.stack([2 * pick, 2 * pick + 1], axis=1).ravel()
        want_cf, want_words = want_cf[keep], want_words[keep]
    assert cf.size == want_cf.size == 2 * min(frames, bench.DUMP_FRAMES)
    assert np.array_equal(cf.view(np.uint32), want_cf.view(np.uint32))
    assert np.array_equal(words.astype(np.int64), want_words.astype(np.int64))
