"""bench.py contract checks that need no GPU: the reference arm prints ONE JSON line with the keys the driver parses, the
CPU arm of config 2 is the reference's own compiled engine where oracle/_ref is present, and our own arm refuses to run
without a GPU instead of falling back to anything; --steps and --dump-outputs are checked without one."""
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]


def _run(*args, timeout=300):
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=timeout,
                          cwd=str(ROOT))


def test_reference_arm_playout_line():
    res = _run("--impl", "reference", "--workload", "playout", "--steps", "1", "--warmup", "1", "--ref-budget", "2")
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "selfplay_positions_per_sec" and d["unit"] == "positions/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1
    assert d["gpu_launches"] == 0
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    cpu = d["cpu_baseline"]
    assert cpu["kind"] in ("reference", "port") and cpu["cores"] >= 1 and cpu["sample"]
    if (ROOT / "oracle" / "_ref" / "ref_playout").exists():
        assert cpu["kind"] == "reference"                       # the reference's own compiled scalar engine


def test_bench_rejects_arguments_it_cannot_honour():
    res = _run("--steps", "0", timeout=60)
    assert res.returncode != 0 and "--steps" in res.stderr
    res = _run("--workload", "playout", "--dump-outputs", "unused", timeout=60)
    assert res.returncode != 0 and "--dump-outputs" in res.stderr
    res = _run("--workload", "eval", "--steps", "3", timeout=60)          # one whole run is the only step it times
    assert res.returncode != 0 and "--steps" in res.stderr


def test_dump_outputs_keeps_a_fixed_sample_under_the_limit(tmp_path):
    """--dump-outputs of a run whose outputs exceed the limit: the same seeded sample of games in every per-game array
    (indices in games.npy), 64-bit sources as float64, the rest as float32, under 64 MB in all."""
    import numpy as np
    import torch

    import bench

    g = torch.Generator().manual_seed(1)
    n = 40_000
    per_game = {"policy": torch.rand((n, 220), generator=g), "legal": torch.rand((n, 220), generator=g) < 0.1,
                "sign": torch.ones((n,), dtype=torch.int8), "phase": torch.randint(0, 8, (n,), generator=g)}
    other = {"outcomes": torch.tensor([3, 4, 5])}
    bench.dump_outputs(str(tmp_path / "a"), per_game, other)
    bench.dump_outputs(str(tmp_path / "b"), per_game, other)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["games.npy", "legal.npy", "outcomes.npy", "phase.npy", "policy.npy", "sign.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64_000_000
    load = {f: (np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)) for f in files}
    assert all(np.array_equal(a, b) for a, b in load.values())
    games = load["games.npy"][0].astype(np.int64)
    assert 0 < games.size < n and np.all(np.diff(games) > 0)
    assert load["policy.npy"][0].dtype == np.float32 and load["phase.npy"][0].dtype == np.float64
    assert np.array_equal(load["policy.npy"][0], per_game["policy"].numpy()[games])
    assert np.array_equal(load["legal.npy"][0], per_game["legal"].numpy()[games].astype(np.float32))
    assert np.array_equal(load["phase.npy"][0], per_game["phase"].numpy()[games].astype(np.float64))
    assert np.array_equal(load["outcomes.npy"][0], [3.0, 4.0, 5.0])


def test_our_arm_needs_a_gpu():
    import torch

    if torch.cuda.is_available():
        return
    res = _run("--steps", "1", "--warmup", "3", timeout=120)
    assert "selfplay_positions_per_sec" not in res.stdout           # no number without the CUDA path
    assert "NVIDIA" in res.stderr or "CUDA" in res.stderr or "cuda" in res.stderr
