"""CPU: the bench.py contract pieces that do not need a GPU - the reference arm's JSON line, the roofline
helpers and the committed ncu summary that feeds `roofline.traffic`."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_reference_arm_prints_one_contract_line(tmp_path):
    """`bench.py --impl reference` times the reference's CPU implementation of the path (here: the oracle port
    of its ATen calls) on a bounded sample of the product arm's workload and prints ONE JSON line; with
    `--dump-outputs` it also writes what its last step computed."""
    import numpy as np

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["gpu_launches"] == 0
    assert d["metric"].startswith("rotation hypotheses scored/sec") and d["unit"] == "hyp*pairs/s"
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] == d["cpu_baseline"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["config"]["pairs"] == 32 and d["config"]["hypotheses_per_gpu"] == 50000      # BASELINE configs[1]
    assert "BASELINE.json configs[1]" in d["config"]["workload"]
    dump = {f.stem: np.load(f) for f in tmp_path.iterdir()}
    assert sorted(dump) == ["R_best", "scores", "topk_idx", "topk_val"]
    assert dump["scores"].shape == (2, 10000) and dump["R_best"].shape == (2, 1, 3, 3)
    assert np.array_equal(dump["topk_idx"][:, 0], dump["scores"].argmax(1))
    assert np.array_equal(dump["topk_val"][:, 0], dump["scores"].max(1))


def test_roofline_inputs():
    import bench

    # algorithmic shared-memory bytes per (pair, hypothesis): 512 voxels x 8 taps x 16 channels x 4 B (SURVEY.md §8d)
    assert bench.GATHER_BYTES_PER_HYP == 512 * 8 * 16 * 4
    peaks = bench.load_peaks()
    assert peaks["hbm_gbs"] > 1000 and peaks["bf16_tflops"] > 100 and "source" in peaks
    traffic = bench.ncu_traffic()          # DRAM bytes per launch of the score kernel from the committed ncu capture
    assert traffic is not None and 1e5 < traffic < 1e9


def test_dump_outputs_writes_npy_within_the_limit(tmp_path):
    """`--dump-outputs`: one .npy per returned tensor; above the size limit a fixed seeded sample of pairs, the
    same one every time, with its pair numbers."""
    import numpy as np
    import torch

    import bench

    t = {"topk_val": torch.randn(1000, 1), "topk_idx": torch.arange(1000.0, dtype=torch.float64)[:, None],
         "R_best": torch.randn(1000, 1, 3, 3)}
    bench.dump_outputs(str(tmp_path / "all"), t)
    for name, x in t.items():
        assert np.array_equal(np.load(tmp_path / "all" / (name + ".npy")), x.numpy())
    assert not (tmp_path / "all" / "rows.npy").exists()
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), t, limit_bytes=4096 + 20_000)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["R_best.npy", "rows.npy", "topk_idx.npy", "topk_val.npy"]
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= 4096 + 20_000
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert rows.dtype == np.float64 and 0 < len(rows) < 1000 and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "topk_idx.npy")[:, 0], rows)
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
