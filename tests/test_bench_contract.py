"""bench.py's JSON contract, checked on the arm that runs without a GPU (--impl reference = the CPU oracle port)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_reference_arm_prints_one_contract_line(tmp_path, oracle):
    import numpy as np
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "Mrays/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["config"]["workload"].startswith("rgbbox 1000x1000 64spp + irreg 1000x1000 64spp")
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # --dump-outputs: the step's frames (rows j % 8 == 0 rendered at 64 spp, the rest zero) as float64
    assert sorted(os.listdir(tmp_path)) == ["irreg.npy", "rgbbox.npy"]
    for name in ("rgbbox", "irreg"):
        got = np.load(tmp_path / f"{name}.npy")
        want, _, _ = oracle.Scene.named(name).prepare(1000, 1000).render(1000, 1000, spp=64, row_start=0, row_step=64)
        assert got.dtype == np.float64 and got.shape == (1000, 1000)
        np.testing.assert_array_equal(got[::64], want[::64])
        assert (got[1::8] == 0).all()


def test_dump_outputs_samples_large_frames_at_fixed_positions(tmp_path):
    """Frames beyond the byte budget are written as the pixels at a seeded sample of positions: the same in every run."""
    import numpy as np
    bench = _bench_module()
    bench.DUMP_BYTES = 8 * 1000
    frame = np.arange(300 * 40, dtype=np.int32).reshape(300, 40) * 1021
    for out in ("a", "b"):
        bench.dump_outputs(str(tmp_path / out), {"big": frame, "small": frame[:5]})
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float64 and a.shape == (500,) and np.array_equal(a, b)
    assert (np.diff(a) > 0).all() and np.isin(a, frame).all()
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "small.npy"), frame[:5])


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=60, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_full_frame_known_answer_helper(oracle):
    """bench.full_frame_equals_oracle (the per-N / per-config `…sha256_equals_oracle…` flags of the JSON line): True for the
    oracle's own frame, False for a frame with one pixel changed, None for a config without a recorded answer."""
    bench = _bench_module()
    frame, _, _ = oracle.render_scene("irreg", 4000, 4000)
    assert bench.full_frame_equals_oracle(frame, "irreg_4000x4000_1spp") is True
    frame[1234, 567] ^= 1
    assert bench.full_frame_equals_oracle(frame, "irreg_4000x4000_1spp") is False
    assert bench.full_frame_equals_oracle(frame, "irreg_123x45_6spp") is None
