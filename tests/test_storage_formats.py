"""Self-play payload files (SURVEY 8b: `run_self_play_worker` + `v1_sharded_shard` / `v1_worker_chunk_manifest` /
`v1_sharded_manifest`; 8f-2 asynchronous writer).  CPU tests: our helpers vs golden vectors produced by the reference's
python (tests/golden/make_storage_golden.py) and -- when oracle/build_ref.py has put the reference's build and python
copy into oracle/_ref -- the reference's own loader opening the files we write.  GPU test: the worker end to end on a
tiny configuration."""
import json
import os
import sys
from pathlib import Path

import pytest
import torch

from liuzhou_b200 import self_play_storage as st
from liuzhou_b200.trajectory_buffer import TensorSelfPlayBatch

GOLDEN = Path(__file__).resolve().parent / "golden" / "storage_formats.json"
REF_DIR = Path(__file__).resolve().parents[1] / "oracle" / "_ref"

PLAN_GRID = [
    dict(total_samples=0, num_shards=4),
    dict(total_samples=1, num_shards=4),
    dict(total_samples=10, num_shards=3),
    dict(total_samples=1000, num_shards=1, target_samples_per_shard=128),
    dict(total_samples=1000, num_shards=3, chunk_target_bytes=2 * 269200, bytes_per_sample=2692),
    dict(total_samples=1000, num_shards=3, target_samples_per_shard=999999, chunk_target_bytes=1, bytes_per_sample=2692),
    dict(total_samples=526857, num_shards=8, chunk_target_bytes=256 << 20, bytes_per_sample=2692),
    dict(total_samples=7, num_shards=100),
    dict(total_samples=4097, num_shards=2, chunk_target_bytes=5000, bytes_per_sample=0),
]

_BUCKETS_A = {str(d): (d + 18) % 5 for d in range(-18, 19)}
_BUCKETS_B = {str(d): (d * d) % 7 for d in range(-18, 19)}
STATS_A = dict(num_games=96, num_positions=11800, black_wins=10, white_wins=7, draws=79, avg_game_length=122.9,
               elapsed_sec=4.0, positions_per_sec=2950.0, games_per_sec=24.0,
               step_timing_ms={"root_puct_ms": 900.0, "finalize_ms": 12.5}, step_timing_ratio={"root_puct_ms": 0.225},
               step_timing_calls={"root_puct_ms": 140}, mcts_counters={"network_evals": 250000},
               piece_delta_buckets=_BUCKETS_A, device="cuda:0")
STATS_B = dict(num_games=32, num_positions=4100, black_wins=1, white_wins=2, draws=29, avg_game_length=128.1,
               elapsed_sec=3.0, positions_per_sec=1366.7, games_per_sec=10.7,
               step_timing_ms={"root_puct_ms": 300.0, "self_play_step_ms": 40.0}, step_timing_ratio={},
               step_timing_calls={"root_puct_ms": 131, "self_play_step_ms": 131}, mcts_counters={"network_evals": 90000, "x": 3},
               piece_delta_buckets=_BUCKETS_B, device="cuda:1", fallback_count=1, fallback_reasons=("graph",))


def synthetic_batch(n: int, seed: int) -> TensorSelfPlayBatch:
    g = torch.Generator().manual_seed(seed)
    states = (torch.rand((n, 11, 6, 6), generator=g) < 0.3).to(torch.float32)
    legal = torch.rand((n, 220), generator=g) < 0.1
    legal[:, 0] = True
    pol = torch.rand((n, 220), generator=g) * legal
    pol = pol / pol.sum(1, keepdim=True)
    value = torch.randint(-1, 2, (n,), generator=g).to(torch.float32)
    soft = torch.tanh(torch.randn((n,), generator=g))
    return TensorSelfPlayBatch(states, legal, pol, value, soft)


def target_vector(seed: int, n: int) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    v = torch.randn((n,), generator=g) * 0.15
    if n > 8:
        v[::5] = 0.0
        v[3] = float("nan")
        v[7] = float("inf")
        v[11 % n] = 1e-7
    return v


def policy_cases():
    """(visits i64[220], priors f32[220], legal bool[220], q f32[220], temperature, beta) -- seeded; ties included."""
    g = torch.Generator().manual_seed(2024)
    cases = []
    for k, (temp, beta) in enumerate([(1.0, 0.0), (0.1, 0.0), (0.0, 0.0), (1.0, 2.0), (0.5, 8.0), (0.0, 3.0), (1.0, 0.5)]):
        legal = torch.rand((220,), generator=g) < 0.12
        legal[k] = True
        visits = torch.randint(0, 6, (220,), generator=g) * legal
        if k % 2 == 0:
            visits[legal.nonzero()[0]] = 5                       # force ties at the maximum
        priors = torch.rand((220,), generator=g) * legal
        priors = priors / priors.sum()
        qv = (torch.randint(-2, 3, (220,), generator=g).float() / 4.0) * (visits > 0)
        cases.append((visits, priors.float(), legal, qv, temp, beta))
    return cases


def test_policy_targets_and_deterministic_choice_match_reference(golden):
    """policy_from_visits (+ beta * priors, target temperature) and the N -> Q -> P -> index move choice of the tree
    backend vs the reference's portable search functions (portable_mcts.py:149-261), batched over the 220-d space."""
    from liuzhou_b200.tree_search import deterministic_action, policy_from_visits

    cases = policy_cases()
    visits = torch.stack([c[0] for c in cases])
    priors = torch.stack([c[1] for c in cases])
    legal = torch.stack([c[2] for c in cases])
    qv = torch.stack([c[3] for c in cases])
    for i, (_, _, _, _, temp, beta) in enumerate(cases):
        got = policy_from_visits(visits[i:i + 1], torch.tensor([temp]), legal=legal[i:i + 1], priors=priors[i:i + 1],
                                 prior_pseudocount=beta)[0]
        want = torch.tensor(golden["policy_targets"][i]["policy"])
        assert torch.allclose(got, want, rtol=1e-5, atol=1e-7), i
        assert float(got[~legal[i]].abs().sum()) == 0.0
    choice = deterministic_action(visits, qv, legal, priors)
    assert choice.tolist() == [g["choice"] for g in golden["policy_targets"]]
    # mixed temperatures in one batch (per-game temperature switch), beta = 0: rows equal their single-row results
    temps = torch.tensor([c[4] for c in cases])
    batch = policy_from_visits(visits, temps)
    for i in range(len(cases)):
        assert torch.equal(batch[i], policy_from_visits(visits[i:i + 1], temps[i:i + 1])[0])


@pytest.fixture(scope="module")
def golden():
    return json.loads(GOLDEN.read_text())


def _eq_batches(a, b):
    for f in ("state_tensors", "legal_masks", "policy_targets", "value_targets", "soft_value_targets"):
        x, y = getattr(a, f), getattr(b, f)
        assert x.dtype == y.dtype and x.shape == y.shape, f
        assert torch.equal(x.cpu(), y.cpu()), f


def test_plan_sample_ranges_golden(golden):
    got = [[list(r) for r in st.plan_sample_ranges(**kw)] for kw in PLAN_GRID]
    assert got == golden["plan"]


def test_target_summaries_golden(golden):
    ours = [st.summarize_scalar_targets(target_vector(seed, n)) for seed, n in ((1, 0), (2, 257), (3, 4099))]
    for o, g in zip(ours, golden["summaries"]):
        assert list(o.keys()) == list(st._ordered_summary(g).keys())
        for k, v in g.items():
            if isinstance(v, int):
                assert o[k] == v, k
            else:
                assert o[k] == pytest.approx(v, rel=1e-5, abs=1e-9), k
    merged = st.merge_target_summaries(golden["summaries"])
    for k, v in golden["summary_merged"].items():
        assert merged[k] == pytest.approx(v, rel=1e-12), k


def test_merge_self_play_stats_golden(golden):
    from liuzhou_b200.self_play import SelfPlayV1Stats
    from liuzhou_b200.self_play_worker import merge_self_play_stats, stats_from_payload

    merged = merge_self_play_stats([SelfPlayV1Stats(**STATS_A), SelfPlayV1Stats(**STATS_B)], elapsed_sec=12.5)
    got, want = merged.to_dict(), golden["stats_merged"]
    assert set(got) == set(want)
    for k, v in want.items():
        if k == "policy_target_audit":
            continue                                   # portable-backend health metric: not produced (DESIGN §8)
        if isinstance(v, dict):
            assert set(got[k]) == set(v), k
            for kk, vv in v.items():
                assert got[k][kk] == pytest.approx(vv, rel=1e-12), (k, kk)
        elif isinstance(v, float):
            assert got[k] == pytest.approx(v, rel=1e-12), k
        else:
            assert got[k] == v, k
    back = stats_from_payload(got)                     # to_dict / from-payload round trip
    assert back.to_dict() == got


def test_sharded_save_matches_reference_layout(golden, tmp_path):
    from liuzhou_b200.self_play import SelfPlayV1Stats

    b = synthetic_batch(1000, 7)
    assert st.estimate_bytes_per_sample(b) == golden["bytes_per_sample"] == 2692
    path = str(tmp_path / "selfplay_iter_001.pt")
    n = st.save_self_play_payload_sharded(path=path, samples=b, stats_payload=SelfPlayV1Stats(**STATS_A).to_dict(),
                                          metadata={"iteration": 1}, num_shards=3, chunk_target_bytes=300 * 2692)
    g = golden["sharded"]
    man = torch.load(path)
    assert n == g["count"] and man["shard_files"] == g["shard_files"] and man["shard_sizes"] == g["shard_sizes"]
    assert sorted(man.keys()) == g["manifest_keys"] and man["avg_bytes_per_sample"] == g["avg_bytes_per_sample"]
    shard0 = torch.load(str(tmp_path / man["shard_files"][0]))
    assert sorted(shard0.keys()) == g["shard_keys"] and sorted(shard0["metadata"].keys()) == g["shard_meta_keys"]
    assert shard0["state_tensors"].untyped_storage().nbytes() == shard0["state_tensors"].numel() * 4   # no staging slack on disk
    loaded, stats, meta = st.load_self_play_payload(path)
    _eq_batches(loaded, b)
    assert meta["loaded_num_samples"] == 1000 and meta["manifest_num_shards"] == n and stats["num_games"] == 96.0
    # DDP-style partial load: shards i % world == rank, in order
    parts = [st.load_self_play_payload(path, ddp_rank=r, ddp_world_size=3)[0] for r in range(3)]
    sizes = man["shard_sizes"]
    for r, p in enumerate(parts):
        assert p.num_samples == sum(s for i, s in enumerate(sizes) if i % 3 == r)
    with pytest.raises(RuntimeError):
        st.load_self_play_payload(path, ddp_rank=5, ddp_world_size=6 + len(sizes))
    with pytest.raises(FileNotFoundError):
        st.load_self_play_payload(str(tmp_path / "missing.pt"))


def test_empty_batch_writes_plain_payload(tmp_path):
    b = synthetic_batch(0, 1)
    path = str(tmp_path / "empty.pt")
    assert st.save_self_play_payload_sharded(path=path, samples=b, stats_payload={}, metadata={}, num_shards=4) == 0
    loaded, _, _ = st.load_self_play_payload(path)
    assert loaded.num_samples == 0


def test_async_writer_surfaces_errors(tmp_path):
    b = synthetic_batch(10, 3)
    blocker = tmp_path / "file"
    blocker.write_text("x")
    w = st.AsyncShardWriter(None)
    w.submit(str(blocker / "sub" / "a.pt"), b, start=0, end=10, stats_payload={}, metadata={})   # parent is a file
    with pytest.raises(RuntimeError):
        w.close()


def _write_fake_worker(tmp_path, widx, batch, stats, prefix):
    """A worker manifest + its chunk files, written exactly the way run_self_play_worker does."""
    from liuzhou_b200.self_play import SelfPlayV1Stats
    from liuzhou_b200.self_play_worker import merge_self_play_stats

    files, sizes = [], []
    with st.AsyncShardWriter(None) as w:
        for lo, hi in st.plan_sample_ranges(total_samples=batch.num_samples, num_shards=1, target_samples_per_shard=150):
            name = f"{prefix}.w{widx:02d}.chunk{len(files):05d}.pt"
            w.submit(str(tmp_path / name), batch, start=lo, end=hi, stats_payload={},
                     metadata={"payload_format": "v1_sharded_shard", "worker_idx": widx})
            files.append(name)
            sizes.append(hi - lo)
    man = {"payload_format": "v1_worker_chunk_manifest", "version": 1, "num_samples": sum(sizes), "num_shards": len(files),
           "shard_files": files, "shard_sizes": sizes, "chunk_target_bytes": 0, "avg_bytes_per_sample": 2692,
           "stats": merge_self_play_stats([SelfPlayV1Stats(**stats)], 1.0).to_dict(),
           "value_target_summary": st.summarize_scalar_targets(batch.value_targets),
           "soft_value_target_summary": st.summarize_scalar_targets(batch.soft_value_targets),
           "mixed_value_target_summary": st.summarize_scalar_targets(st.mixed_value_targets(batch, 0.25)),
           "metadata": {"worker_idx": widx}}
    p = str(tmp_path / f"worker_manifest_{widx:02d}.pt")
    torch.save(man, p)
    return p


def test_worker_manifest_merge_and_reference_loader(tmp_path):
    from liuzhou_b200.self_play_worker import merge_worker_manifests

    b0, b1 = synthetic_batch(400, 11), synthetic_batch(333, 12)
    m0 = _write_fake_worker(tmp_path, 0, b0, STATS_A, "selfplay_iter_002")
    m1 = _write_fake_worker(tmp_path, 1, b1, STATS_B, "selfplay_iter_002")
    out = str(tmp_path / "selfplay_iter_002.pt")
    merged, v, s, m, n_files = merge_worker_manifests([m0, m1], output_path=out, metadata_base={"iteration": 2},
                                                      target_samples_per_shard=150, chunk_target_bytes=0, elapsed_sec=9.0)
    assert merged.num_games == 128 and merged.num_positions == 15900 and n_files == 3 + 3
    assert v["total"] == 733 and m["total"] == 733 and s["finite_count"] == 733
    man = torch.load(out)
    assert man["payload_format"] == "v1_sharded_manifest" and man["num_samples"] == 733
    assert man["metadata"]["value_target_summary"]["total"] == 733
    loaded, stats, meta = st.load_self_play_payload(out)
    _eq_batches(loaded, st.concat_batches([b0, b1]))          # worker-major, chunk order
    if not (REF_DIR / "pysrc" / "v1").is_dir():
        pytest.skip("oracle/_ref/pysrc not present: cross-loading by the reference's own loader skipped")
    saved_path = list(sys.path)
    sys.path[:0] = [str(REF_DIR / "pysrc"), str(REF_DIR)]
    try:
        import v1.train as T
        from v1.python.self_play_types import SelfPlayV1Stats as RefStats
        from v1.python.trajectory_buffer import TensorSelfPlayBatch as RefBatch
    finally:
        sys.path[:] = saved_path
    ref_batch, ref_stats, ref_meta = T._load_self_play_payload(out)
    _eq_batches(ref_batch, loaded)
    assert ref_stats == stats and ref_meta["loaded_num_samples"] == 733
    part, _, _ = T._load_self_play_payload(out, ddp_rank=1, ddp_world_size=2)
    ours, _, _ = st.load_self_play_payload(out, ddp_rank=1, ddp_world_size=2)
    _eq_batches(part, ours)
    # and the reverse direction: a manifest written by the reference opens with our loader
    ref_path = str(tmp_path / "ref_written.pt")
    T._save_self_play_payload_sharded(path=ref_path, samples=RefBatch(*(getattr(b0, f) for f in st._FIELDS)),
                                      stats=RefStats(**STATS_A), metadata={}, num_shards=2)
    back, _, _ = st.load_self_play_payload(ref_path)
    _eq_batches(back, b0)


def test_stable_init_matches_reference(golden):
    """Same seed -> bit-identical bootstrap weights as the reference's `_init_model_stable_resnet` on its ChessNet."""
    import hashlib

    from liuzhou_b200.net import ChessNet
    from liuzhou_b200.selfplay_stage import init_model_stable_resnet

    torch.manual_seed(999)
    before = torch.random.get_rng_state()
    net = ChessNet()
    torch.random.set_rng_state(before)
    init_model_stable_resnet(net, seed=20260314)
    assert torch.equal(torch.random.get_rng_state(), before)             # ambient RNG state restored
    h = hashlib.sha256()
    for k, v in net.state_dict().items():
        h.update(k.encode())
        h.update(v.detach().cpu().contiguous().numpy().tobytes())
    assert h.hexdigest() == golden["stable_init_sha256"]
    with pytest.raises(ValueError):
        init_model_stable_resnet(net, seed=0)


def test_stage_cli_accepts_big_train_flags(tmp_path):
    """The flag list scripts/big_train_v1.sh:667-700 passes for --stage selfplay parses; other stages' flags are ignored."""
    from liuzhou_b200 import selfplay_stage as S

    argv = ["--pipeline", "v1", "--stage", "selfplay", "--device", "cuda:0", "--devices", "cuda:0,cuda:1,cuda:1",
            "--train_devices", "cuda:0", "--infer_devices", "cuda:0", "--self_play_games", "32768", "--mcts_simulations", "800",
            "--temperature_init", "1.0", "--temperature_final", "0.1", "--temperature_threshold", "10",
            "--exploration_weight", "1.0", "--dirichlet_alpha", "0.3", "--dirichlet_epsilon", "0.25", "--soft_value_k", "2.0",
            "--soft_label_alpha", "0.25", "--max_game_plies", "512", "--self_play_concurrent_games", "4096",
            "--self_play_opening_random_moves", "4", "--sparse_ply", "1", "--sparse_top_k", "8", "--self_play_backend", "process",
            "--self_play_target_samples_per_shard", "0", "--self_play_chunk_target_bytes", "268435456",
            "--model_init_seed", "20260314", "--checkpoint_dir", str(tmp_path), "--self_play_output", str(tmp_path / "sp.pt"),
            "--self_play_iteration_seed", "7", "--self_play_stats_json", str(tmp_path / "sp.json")]
    args, ignored = S.build_parser().parse_known_args(argv)
    assert ignored == ["--train_devices", "cuda:0", "--infer_devices", "cuda:0"]
    assert args.self_play_games == 32768 and args.self_play_chunk_target_bytes == 268435456 and args.self_play_sample_moves
    assert S.parse_device_list(args.device, args.devices) == ["cuda:0", "cuda:1"]
    assert S._resolve_seeds(args) == (7, 20260314)
    with pytest.raises(RuntimeError):
        S.parse_device_list("cpu", None)                                  # no CPU path
    args.self_play_iteration_seed = -3
    with pytest.raises(ValueError):
        S._resolve_seeds(args)
    # checkpoint loader: `model_state_dict` wrapper and bare state dicts
    from liuzhou_b200.net import ChessNet
    a, b = ChessNet(), ChessNet()
    torch.save({"model_state_dict": a.state_dict(), "iteration": 3}, str(tmp_path / "ck.pt"))
    S.load_checkpoint_into_model(b, str(tmp_path / "ck.pt"))
    assert all(torch.equal(x, y) for x, y in zip(a.state_dict().values(), b.state_dict().values()))
    with pytest.raises(FileNotFoundError):
        S.load_checkpoint_into_model(b, str(tmp_path / "none.pt"))


@pytest.mark.gpu
def test_stage_cli_end_to_end(tmp_path):
    """`python -m liuzhou_b200.selfplay_stage` on one GPU: manifest + stats JSON as the next stage expects them."""
    import subprocess

    out, js = tmp_path / "run" / "selfplay_iter_001.pt", tmp_path / "run" / "selfplay_iter_001.json"
    cmd = [sys.executable, "-m", "liuzhou_b200.selfplay_stage", "--stage", "selfplay", "--device", "cuda:0",
           "--self_play_games", "96", "--mcts_simulations", "16", "--self_play_concurrent_games", "64", "--max_game_plies", "48",
           "--self_play_output", str(out), "--self_play_iteration_seed", "1", "--self_play_stats_json", str(js),
           "--self_play_target_samples_per_shard", "1500", "--batch_size", "256"]
    r = subprocess.run(cmd, cwd=str(Path(__file__).resolve().parents[1]), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    rep = json.loads(js.read_text())
    assert rep["num_games"] == 96.0 and rep["self_play_iteration_seed"] == 1 and rep["piece_delta_bucket_total"] == 96
    assert rep["value_target_summary"]["total"] == int(rep["num_positions"])
    batch, stats, meta = st.load_self_play_payload(str(out))
    assert batch.num_samples == int(rep["num_positions"]) and meta["stage"] == "selfplay" and meta["self_play_games"] == 96


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["cuda_root", "portable"])
def test_run_self_play_worker_end_to_end(tmp_path, backend):
    from liuzhou_b200.net import ChessNet
    from liuzhou_b200.self_play_worker import run_self_play_iteration, run_self_play_worker

    torch.manual_seed(5)
    model = ChessNet()
    state_path = str(tmp_path / "model_state_cpu.pt")
    torch.save({k: v.detach().cpu() for k, v in model.state_dict().items()}, state_path)
    kw = dict(mcts_simulations=16, temperature_init=1.0, temperature_final=0.1, temperature_threshold=10,
              exploration_weight=1.0, dirichlet_alpha=0.3, dirichlet_epsilon=0.25, soft_value_k=2.0,
              opening_random_moves=2, max_game_plies=64, concurrent_games_per_device=64, search_backend=backend)
    man_path = str(tmp_path / "worker_manifest.pt")
    row = run_self_play_worker(worker_idx=0, shard_device="cuda:0", shard_games=160, seed=99, model_state_path=state_path,
                               output_path=man_path, chunk_output_dir=str(tmp_path), chunk_file_prefix="sp.w00",
                               target_samples_per_shard=2000, soft_label_alpha=0.25, **kw)
    man = torch.load(man_path)
    assert man["payload_format"] == "v1_worker_chunk_manifest" and row["num_samples"] == man["num_samples"] > 0
    assert man["metadata"]["num_selfplay_batches"] == 3 and man["stats"]["num_games"] == 160.0      # 64 + 64 + 32 games
    assert sum(man["shard_sizes"]) == man["num_samples"] == int(man["stats"]["num_positions"])
    assert man["value_target_summary"]["total"] == man["num_samples"] and man["value_target_summary"]["nonfinite_count"] == 0
    rows = 0
    for name, size in zip(man["shard_files"], man["shard_sizes"]):
        shard = torch.load(os.path.join(str(tmp_path), name))
        assert shard["metadata"]["payload_format"] == "v1_sharded_shard" and shard["state_tensors"].shape == (size, 11, 6, 6)
        assert shard["legal_masks"].dtype == torch.bool and shard["policy_targets"].shape == (size, 220)
        assert torch.isfinite(shard["value_targets"]).all() and torch.isfinite(shard["soft_value_targets"]).all()
        # every stored policy is a distribution over that row's legal actions
        assert torch.all((shard["policy_targets"] > 0) <= shard["legal_masks"])
        assert torch.allclose(shard["policy_targets"].sum(1), torch.ones(size), atol=1e-4)
        rows += size
    assert rows == man["num_samples"]
    # iteration-level driver (world size 1): emits the v1_sharded_manifest the trainer opens
    out = str(tmp_path / "iter" / "selfplay_iter_003.pt")
    res = run_self_play_iteration(model, num_games=96, iteration_seed=3, output_path=out, metadata_base={"iteration": 3}, **kw)
    merged_stats = res[0]
    batch, stats, meta = st.load_self_play_payload(out, device="cuda:0")
    assert batch.num_samples == merged_stats.num_positions == int(stats["num_positions"]) and batch.state_tensors.is_cuda
    assert meta["iteration"] == 3 and merged_stats.num_games == 96
