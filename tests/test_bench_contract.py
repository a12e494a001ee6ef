"""CPU test of bench.py's contract for the arm that can run without a GPU: `--impl reference` (the CPU port
of the path, oracle/).  One JSON line with the keys the driver parses; values self-consistent.
GPU test of --dump-outputs: what the default arm's last timed step computed, the same on every run."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys(oracle_lib):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1",
                          "--steps", "1", "--warmup", "1"], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "geodesic maps/sec" and d["unit"] == "maps/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["data"] == "synthetic"
    assert d["dtype"] == "f32" and d["vs_baseline"] is None and d["scaling"] == "weak"
    cfg = d["config"]
    assert cfg["N"] == 50000 and cfg["Q"] == 128 and cfg["k"] == 8 and cfg["max_step"] == 32 and "workload" in cfg
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == "maps/s"
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    # value = maps per second of one scene's worth of seeds
    assert abs(d["value"] - cfg["Q"] / (d["ms_per_step"] * 1e-3)) <= 1e-6 * d["value"]


def test_bench_refuses_to_run_the_product_arm_without_a_gpu():
    import torch

    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--no-e2e",
                          "--no-cpu-baseline"], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert out.returncode != 0 and "no CUDA device" in (out.stderr + out.stdout)


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["c1", "c2"])
def test_dump_outputs_are_the_last_timed_step(tmp_path, cuda_lib, workload):
    """--steps 3: exactly one timed call of scenes 0, 1, 2 of the workload; the dump holds scene 2's seeds and maps
    (all columns at c1, a fixed sample of them at c2), bit-identical between two runs and to a direct call"""
    import numpy as np
    import torch

    from geoformer_b200.guidance import geodesic_guidance
    from geoformer_b200.scenes import CONFIGS, scene

    dumps = []
    for run in range(2):
        out_dir = tmp_path / str(run)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", "3",
                              "--warmup", "1", "--no-e2e", "--no-cpu-baseline", "--no-extras", "--dump-outputs",
                              str(out_dir)], cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        d = json.loads([l for l in out.stdout.splitlines() if l.strip().startswith("{")][-1])
        assert d["steps"] == 3 and d["repeats"] == 1 and len(d["repeats_ms"]) == 1
        assert d["pipeline"]["scenes_per_call"] * d["pipeline"]["calls_per_region"] == 3
        assert sorted(os.listdir(out_dir)) == ["geo.npy", "geo_columns.npy", "seeds.npy"]
        assert sum(os.path.getsize(out_dir / f) for f in os.listdir(out_dir)) <= 64 << 20
        dumps.append({f[:-4]: np.load(out_dir / f) for f in os.listdir(out_dir)})
    for name, a in dumps[0].items():
        assert a.dtype in (np.float32, np.float64), name
        assert np.array_equal(a, dumps[1][name]), name
    cfg = CONFIGS[workload]
    seeds, geo = geodesic_guidance(scene(cfg["n"], cfg["seed"] + 2).cuda(), cfg["Q"], cfg["k"], cfg["radius"],
                                   cfg["max_step"])
    cols = dumps[0]["geo_columns"].astype(np.int64)
    assert len(cols) == (cfg["n"] if workload == "c1" else 32768)
    assert np.array_equal(dumps[0]["seeds"], seeds.cpu().numpy().astype(np.float64))
    assert np.array_equal(dumps[0]["geo"], geo[:, torch.from_numpy(cols).cuda()].cpu().numpy())
