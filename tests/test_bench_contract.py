"""bench.py's reference arm (--impl reference) end to end on the CPU: one JSON line on stdout with the keys the driver reads.
The arm times the UNMODIFIED reference (oracle/_ref) where it travelled, else the C oracle; here on the tiny config so that the
whole test takes seconds (BARK_B200_BENCH_CONFIG=tiny; every real run uses bark-small)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, BARK_B200_BENCH_CONFIG="tiny", BARK_B200_QUIET="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-800:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[-800:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "audio_s/s" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None
    assert d["metric"].startswith("audio sec/sec")
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, BARK_B200_BENCH_CONFIG="tiny", RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_are_reproducible(tmp_path):
    """--dump-outputs writes the last timed step's waveform and token ids as float32 .npy files; the same arguments give the
    same inputs, so two runs write the same arrays."""
    import numpy as np
    env = dict(os.environ, BARK_B200_BENCH_CONFIG="tiny", BARK_B200_QUIET="1")
    dumps = []
    for run in ("a", "b"):
        d = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0",
                            "--dump-outputs", str(d)], capture_output=True, text=True, env=env, timeout=600)
        assert r.returncode == 0, r.stderr[-800:]
        dumps.append({p.stem: np.load(p) for p in sorted(d.glob("*.npy"))})
    assert sorted(dumps[0]) == ["audio", "coarse_tokens", "fine_tokens", "semantic_tokens"]
    for name, a in dumps[0].items():
        assert a.dtype == np.float32 and a.size > 0, name
        assert np.array_equal(a, dumps[1][name]), name
