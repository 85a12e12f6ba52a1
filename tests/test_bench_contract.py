"""bench.py's reference arm runs without a GPU (it times the oracle): its one JSON line must carry the contract's keys and
say what it ran.  --dump-outputs writes what the timed path computed in its last step, the same from run to run, on
both arms (the b200 arm's test needs a B200)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--frames-per-link", "4"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1                                            # ONE JSON line on stdout
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "Msamples/s" and d["higher_is_better"] is True and d["gpu_launches"] == 0
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == (os.cpu_count() or 1) and cb["value"] == d["value"]
    # the line states what was run: the links and frames of this run, not the b200 arm's
    cfg = d["config"]
    assert cfg["links_per_gpu"] == cb["cores"] and cfg["frames_per_link"] == 4 and "bounded_sample_of" in cfg
    n_samples = cfg["links_per_gpu"] * (128 + 4 * (4961 + 1100))
    assert cfg["samples_per_gpu"] == n_samples and str(n_samples) in cb["sample"]
    assert d["crc_ok_per_step"] >= d["frames_per_step"] - 2           # 64-QAM 3/4 at 30 dB


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_steps_must_be_at_least_one():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr and out.stdout.strip() == ""


def _dump(out_dir, args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args + ["--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    files = sorted(os.listdir(out_dir))
    assert sum(os.path.getsize(os.path.join(out_dir, f)) for f in files) <= 64 << 20
    return json.loads(out.stdout), {f[:-4]: np.load(os.path.join(out_dir, f)) for f in files}


def _check_dump(line, a, n_sent):
    """The dump is the frame table and PSDU bytes of the line's last step: every CRC-ok frame's bytes are a PSDU that was
    sent (bench.make_psdus with the arms' seed 1000)."""
    import bench
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    n = line["frames_per_step"]
    assert np.array_equal(a["frame_index"], np.arange(n)) and np.array_equal(a["psdu_index"], np.arange(n))
    assert a["psdu_bytes"].shape == (n, bench.PSDU_MAX)
    for k in ("trigger", "link", "sig_ok", "length", "crc_ok", "snr", "psdu_off"):
        assert a["frame_" + k].shape == (n,), k
    assert int(a["frame_crc_ok"].sum()) == line["crc_ok_per_step"] > 0
    sent = set(bench.make_psdus(n_sent, 1000))
    for i in np.nonzero(a["frame_crc_ok"])[0]:
        ln, row = int(a["frame_length"][i]), a["psdu_bytes"][i]
        assert bytes(row[:ln].astype(np.uint8)) in sent and (row[ln:] == -1).all(), i


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


def test_reference_arm_dumps_its_last_step(tmp_path):
    args = ["--impl", "reference", "--steps", "2", "--warmup", "0", "--frames-per-link", "3"]
    line, a = _dump(tmp_path / "a", args)
    _check_dump(line, a, line["config"]["links_per_gpu"] * 3)
    _same(a, _dump(tmp_path / "b", args)[1])


@pytest.mark.gpu
def test_b200_arm_dumps_its_last_step(tmp_path):
    args = ["--links", "2", "--frames-per-link", "24", "--steps", "3", "--warmup", "1", "--no-e2e", "--no-cpu", "--no-time-shard"]
    line, a = _dump(tmp_path / "a", args)
    assert line["steps"] == 3
    _check_dump(line, a, 2 * 24)
    _same(a, _dump(tmp_path / "b", args)[1])
