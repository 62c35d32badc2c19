#!/usr/bin/env python3
"""bench.py -- headline benchmark of the liuzhou_b200 hot path (contract: see README / DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload selfplay|playout] [--impl ours|reference]
                    [--dump-outputs DIR]

N > 1 is launched by the driver through torchrun (one rank per GPU, NCCL); games are independent, so ranks
shard the games with no data-path collective ("scaling": "weak").  Rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

SEED = 20260314  # reference stable-init seed (scripts/big_train_v1.sh:24)


# ----------------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------------
def measured_peaks() -> tuple[dict, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return json.loads(p.read_text()), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int = 0):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines: list[str] = []
        self._thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu_index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.lines.append(line.strip())
        self._thread = threading.Thread(target=pump, daemon=True)
        self._thread.start()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2])); power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def dist_setup(n_gpus: int):
    import torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(0)
        local_rank = 0
    return world, rank, local_rank


def barrier_sync(world: int):
    import torch

    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(value: float, world: int) -> float:
    if world <= 1:
        return value
    import torch
    import torch.distributed as dist

    t = torch.tensor([value], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def all_ranks(value: float, world: int) -> list:
    """The value of every rank, in rank order (diagnostic next to the max the metric is computed from)."""
    if world <= 1:
        return [value]
    import torch
    import torch.distributed as dist

    t = torch.tensor([value], dtype=torch.float64, device="cuda")
    out = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return [float(x.item()) for x in out]


def sum_over_ranks(value: float, world: int) -> float:
    if world <= 1:
        return value
    import torch
    import torch.distributed as dist

    t = torch.tensor([value], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


class L2Flusher:
    """Writes a buffer larger than the 126 MB L2 between timed iterations."""

    def __init__(self, device, mib: int = 256):
        import torch

        self.buf = torch.empty((mib << 20,), dtype=torch.uint8, device=device)

    def flush(self):
        self.buf.add_(1)


DUMP_LIMIT_BYTES = 60 << 20          # array data; with the .npy headers a dump stays under 64 MB (64e6 bytes)


def dump_outputs(out_dir: str, per_game: dict, other: dict) -> None:
    """--dump-outputs: write what the timed path computed as DIR/<name>.npy -- float64 for 64-bit sources, float32
    otherwise (exact for every array dumped here) -- so that two builds can be compared output for output.  The arrays
    of `per_game` share their first dimension (the game); if everything would exceed DUMP_LIMIT_BYTES, the same fixed,
    seeded sample of games is kept in each of them and its indices are written as games.npy."""
    import numpy as np
    import torch

    def host(t):
        wide = t.dtype in (torch.int64, torch.float64)
        return t.detach().to("cpu", torch.float64 if wide else torch.float32).numpy()

    rows = {k: host(v) for k, v in per_game.items()}
    rest = {k: host(v) for k, v in other.items()}
    n = next(iter(rows.values())).shape[0]
    row_bytes = sum(a[0].nbytes for a in rows.values())
    keep = (DUMP_LIMIT_BYTES - sum(a.nbytes for a in rest.values())) // (row_bytes + 8)
    if keep < n:
        games = np.sort(np.random.default_rng(SEED).choice(n, keep, replace=False))
        rows = {k: a[games] for k, a in rows.items()}
        rest["games"] = games.astype(np.float64)
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for k, a in {**rows, **rest}.items():
        np.save(out / f"{k}.npy", a)


def reference_gpu_line(games: int, sims: int, device_index: int, timeout_s: float = 600.0) -> dict:
    """The v1 REFERENCE on the same GPU, same games / sims / network: the reference's own unmodified python
    (`self_play_v1_gpu`, v1/python/self_play_gpu_runner.py:21-307 -> `V1RootMCTS.search_batch`, mcts_gpu.py:1249-1457)
    over its own `v0_core` CUDA extension (oracle/_ref: its three .cu kernels compiled for sm_100 from the unmodified
    sources) with its own PyTorch ChessNet under fp16 autocast -- run by oracle/ref_runner.py in a process of its own
    (a process holds one module named v0_core).  This is the denominator of north_star's ">= 100x the v1 reference's
    positions/s per GPU" and is reported next to our drop-in of the same backend (`root_puct_backend`)."""
    runner = ROOT / "oracle" / "ref_runner.py"
    if not (ROOT / "oracle" / "_ref" / "pysrc").is_dir() or not list((ROOT / "oracle" / "_ref").glob("v0_core*.so")):
        return {"unavailable": "oracle/_ref (reference binaries + python copy) not present on this box"}
    cmd = [sys.executable, str(runner), "selfplay", "--v0core", "ref", "--games", str(games), "--sims", str(sims),
           "--device", f"cuda:{device_index}", "--warmup-games", str(min(256, games)), "--seed", str(SEED + 1)]
    try:
        res = subprocess.run(cmd, cwd=str(ROOT), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                             timeout=timeout_s)
    except subprocess.TimeoutExpired:
        return {"unavailable": f"reference run exceeded {timeout_s:.0f}s"}
    if res.returncode != 0:
        return {"unavailable": "reference run failed: " + res.stderr.strip().splitlines()[-1][:300] if res.stderr.strip() else "rc != 0"}
    out = json.loads(res.stdout.strip().splitlines()[-1])
    return {"value": out["positions_per_sec"], "unit": "positions/s", "positions": out["positions"],
            "seconds": out["seconds"], "e2e": {"value": out["e2e_positions_per_sec"], "unit": "positions/s",
                                               "d2h_bytes_per_step": out["d2h_bytes"]},
            "avg_game_length": out["avg_game_length"], "draws": out["draws"],
            "what": "UNMODIFIED reference python + reference v0_core CUDA (sm_100) + reference ChessNet (PyTorch eager, fp16 "
                    f"autocast), {games} games x {sims} sims, search_backend=cuda_root, same GPU, separate process"}


def legacy_cpu_line(timeout_s: float = 180.0) -> dict:
    """BASELINE configs[0]: the legacy `src/` python rule engine + `src/mcts.py::self_play`, 1 game, 64 sims/move, the
    reference tests' small random-init net, on ONE host core (the code is single-threaded python)."""
    runner = ROOT / "oracle" / "ref_runner.py"
    if not (ROOT / "oracle" / "_ref" / "pysrc" / "src" / "mcts.py").exists():
        return {"unavailable": "oracle/_ref/pysrc not present on this box"}
    try:
        res = subprocess.run([sys.executable, str(runner), "legacy", "--games", "1", "--sims", "64"], cwd=str(ROOT),
                             stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout_s)
    except subprocess.TimeoutExpired:
        return {"unavailable": f"legacy run exceeded {timeout_s:.0f}s"}
    if res.returncode != 0:
        return {"unavailable": "legacy run failed"}
    out = json.loads(res.stdout.strip().splitlines()[-1])
    return {"value": out["positions_per_sec"], "unit": "positions/s", "sims_per_sec": out["sims_per_sec"],
            "positions": out["positions"], "seconds": out["seconds"], "cores": 1, "kind": "reference",
            "what": "BASELINE configs[0]: legacy src/ rule engine + src/mcts.py self_play, 1 game x 64 sims, tiny net, CPU"}


def ncu_dram_traffic(kernel_substr: str):
    """(bytes per launch, csv name): dram__bytes_read.sum + dram__bytes_write.sum of the newest committed
    `profiles/r*_ncu_full.csv` summary that has a row for the kernel (ncu --set full capture of the bench command)."""
    import csv
    import re

    best = None
    for f in sorted((ROOT / "profiles").glob("r*ncu_full*.csv")):
        try:
            rows = list(csv.reader(f.open()))
        except Exception:
            continue
        if len(rows) < 3 or "Kernel Name" not in rows[0]:
            continue
        h = rows[0]
        try:
            ki, ri, wi = h.index("Kernel Name"), h.index("dram__bytes_read.sum"), h.index("dram__bytes_write.sum")
        except ValueError:
            continue
        unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        vals = [(float(r[ri]) * unit.get(rows[1][ri], 1.0) + float(r[wi]) * unit.get(rows[1][wi], 1.0))
                for r in rows[2:] if len(r) > max(ki, ri, wi) and kernel_substr in r[ki]]
        if vals:
            rnd = int(re.match(r"r(\d+)", f.name).group(1)) if re.match(r"r(\d+)", f.name) else 0
            cand = (rnd, f.stat().st_mtime, sum(vals) / len(vals), f.name)
            if best is None or cand[:2] > best[:2]:
                best = cand
    return (best[2], "profiles/" + best[3]) if best else (None, None)


# ----------------------------------------------------------------------------------------------------
# workload: config 2 -- rule-engine-only random playouts, 65,536 concurrent games per GPU
# ----------------------------------------------------------------------------------------------------
PLAYOUT_GAMES = 65_536
PLAYOUT_BYTES_PER_PLY = 72   # SURVEY.md section 8d: 32 B state read + 32 B write + 8 B RNG / cursor


def cpu_playout_baseline(budget_s: float = 12.0, threads: int | None = None) -> dict:
    """Oracle port (plain C restatement of the v0 C++ scalar engine loop) on the host cores; bounded sample."""
    import oracle
    from concurrent.futures import ThreadPoolExecutor

    cores = threads or os.cpu_count() or 1
    oracle.lib()
    chunk = 256
    t0 = time.perf_counter()
    plies = games = 0
    next_game = 0
    with ThreadPoolExecutor(max_workers=cores) as pool:
        while time.perf_counter() - t0 < budget_s and next_game < PLAYOUT_GAMES:
            futs = [pool.submit(oracle.random_playouts_range, SEED, next_game + i * chunk, next_game + (i + 1) * chunk)
                    for i in range(cores)]
            next_game += cores * chunk
            for f in futs:
                r = f.result()
                plies += r["plies"]
                games += chunk
    dt = time.perf_counter() - t0
    return {"value": plies / dt, "unit": "positions/s", "cores": cores, "kind": "port",
            "sample": f"{games} of {PLAYOUT_GAMES} games ({plies} plies) of the same seeded workload in {dt:.1f}s, "
                      f"oracle/lz_oracle.c scalar-engine loop, {cores} threads"}


def ref_engine_playout_baseline(budget_s: float = 10.0, threads: int | None = None) -> dict:
    """The reference's OWN scalar engine (rule_engine.cpp / move_generator.cpp / game_state.cpp compiled from its
    unmodified sources by oracle/build_ref.py, driven by oracle/ref_playout_harness.cpp) playing uniform-random games --
    v0::GenerateAllLegalMoves + v0::ApplyMove per ply -- on all host threads for a bounded wall-clock sample."""
    exe = ROOT / "oracle" / "_ref" / "ref_playout"
    if not exe.exists():
        return {"unavailable": "oracle/_ref/ref_playout not present on this box"}
    import subprocess
    cores = threads or os.cpu_count() or 1
    try:
        res = subprocess.run([str(exe), str(cores), f"{budget_s:.1f}", str(SEED)], capture_output=True, text=True,
                             timeout=budget_s * 3 + 30)
        r = json.loads(res.stdout.strip().splitlines()[-1])
    except Exception as exc:  # pragma: no cover
        return {"unavailable": f"ref_playout failed: {exc!r}"[:200]}
    return {"value": r["plies_per_sec"], "unit": "positions/s", "cores": cores, "kind": "reference",
            "sample": f"{r['games']} uniform-random games ({r['plies']} plies) in {r['seconds']:.1f}s: the reference's compiled "
                      f"scalar engine (v0::GenerateAllLegalMoves + v0::ApplyMove per ply), {cores} threads"}


def run_playout(args, world, rank, local_rank):
    import torch

    from liuzhou_b200 import _lib, native

    dev = torch.device("cuda", local_rank)
    peaks, peak_kind = measured_peaks()
    games = PLAYOUT_GAMES
    pb = native.PlayoutBatch(games, seed=SEED, device=dev, game_offset=rank * games)
    flusher = L2Flusher(dev)
    stream = torch.cuda.current_stream(dev)

    def step():
        pb.reset()
        pb.run()

    for _ in range(args.warmup):
        step()
        flusher.flush()
    barrier_sync(world)
    launches0 = _lib.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    kernel_ms = []
    total_plies = 0
    t_step = []
    for _ in range(args.steps):
        flusher.flush()
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record(stream)
        pb.reset()
        e1.record(stream)
        pb.run()
        e2.record(stream)
        e2.synchronize()
        t_step.append(e0.elapsed_time(e2))
        kernel_ms.append(e1.elapsed_time(e2))
        total_plies += int(pb.plies.sum().item())
    barrier_sync(world)
    clocks = sampler.stop() if rank == 0 else {}
    launches = _lib.launch_count() - launches0
    elapsed_ms = max_over_ranks(sum(t_step), world)
    all_plies = sum_over_ranks(float(total_plies), world)
    value = all_plies / (elapsed_ms / 1e3)

    # e2e: the same pass through the public API with HOST buffers: initial states (reference byte layout) are
    # copied from pinned host memory, packed, played, unpacked and the final states + results copied back.
    st_host = [t.cpu().pin_memory() for t in native.unpack_states(native.init_states(games, dev))]
    out_host = [torch.empty_like(t).pin_memory() for t in st_host]
    res_host = torch.empty((games,), dtype=torch.int8).pin_memory()
    ply_host = torch.empty((games,), dtype=torch.int32).pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in st_host)
    d2h = h2d + res_host.numel() + ply_host.numel() * 4
    e2e_ms, e2e_plies = [], 0
    for it in range(args.warmup + args.steps):
        flusher.flush()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dev_st = [t.to(dev, non_blocking=True) for t in st_host]
        pb.packed = native.pack_states(dev_st)
        pb.plies.zero_(); pb.result.fill_(2)
        pb.run()
        for dst, src in zip(out_host, native.unpack_states(pb.packed)):
            dst.copy_(src, non_blocking=True)
        res_host.copy_(pb.result, non_blocking=True)
        ply_host.copy_(pb.plies, non_blocking=True)
        torch.cuda.synchronize()
        if it >= args.warmup:
            e2e_ms.append((time.perf_counter() - t0) * 1e3)
            e2e_plies += int(ply_host.sum())
    e2e_elapsed = max_over_ranks(sum(e2e_ms), world)
    e2e_value = sum_over_ranks(float(e2e_plies), world) / (e2e_elapsed / 1e3)

    if rank != 0:
        return None
    k_ms = sum(kernel_ms) / len(kernel_ms)
    plies_per_launch = total_plies / args.steps
    achieved = plies_per_launch * PLAYOUT_BYTES_PER_PLY / (k_ms / 1e3) / 1e9
    cpu_port = cpu_playout_baseline()
    cpu = ref_engine_playout_baseline()
    if "unavailable" in cpu:                    # no reference binary on this box: the oracle port stands in
        cpu = cpu_port
    return {
        "metric": "selfplay_positions_per_sec", "value": value, "unit": "positions/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "rule_engine_random_playouts (BASELINE configs[1])", "games_per_gpu": games,
                   "policy": "uniform random (counter-based RNG), 0 MCTS sims", "max_game_plies": 512,
                   "seed": SEED, "l2": "256 MiB buffer rewritten between timed iterations"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "positions/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": achieved / peaks["hbm_gbs"], "traffic": None, "peak_kind": peak_kind,
                     "kernel": "playout_kernel", "kernel_ms": k_ms,
                     "algorithmic_bytes_per_unit": PLAYOUT_BYTES_PER_PLY, "units_per_launch": plies_per_launch},
        "cpu_baseline": cpu,
        "cpu_port": cpu_port,
    }


def run_reference_playout(args):
    """--impl reference for the playout workload: the CPU engine on all host threads, bounded sample per step."""
    per_step = max(1.0, min(10.0, min(60.0, float(args.ref_budget)) / max(1, args.steps + args.warmup)))
    vals = []
    last = None
    for it in range(args.warmup + args.steps):
        last = ref_engine_playout_baseline(budget_s=per_step)
        if "unavailable" in last:
            last = cpu_playout_baseline(budget_s=per_step)
        if it >= args.warmup:
            vals.append(last["value"])
    value = sum(vals) / len(vals)
    last["value"] = value
    return {
        "impl": "reference", "metric": "selfplay_positions_per_sec", "value": value, "unit": "positions/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i8", "data": "synthetic",
        "config": {"workload": "rule_engine_random_playouts (BASELINE configs[1])", "games_per_gpu": PLAYOUT_GAMES,
                   "seed": SEED},
        "cpu_baseline": last,
        "e2e": {"value": value, "unit": "positions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


# ----------------------------------------------------------------------------------------------------
# workload: config 3 -- wave-batched MCTS self-play, 4,096 games x 200 sims/move, default net bf16 (per GPU)
# ----------------------------------------------------------------------------------------------------
SELFPLAY_GAMES = 4096
SELFPLAY_SIMS = 200


def _default_model():
    import torch

    from liuzhou_b200.net import ChessNet

    torch.manual_seed(SEED)
    return ChessNet()


class CpuSelfPlaySession:
    """The reference's own CPU tree search (oracle/_ref/_liuzhou_portable_cpp: threaded C++ `PortableTreeBatch`, the
    reference's `--search_backend portable --portable_mcts_backend cpp`) + the fp32 PyTorch network on all host cores,
    as ONE continuous self-play session: `trees` concurrent games (every network call is a batch of up to `trees`
    leaves), `sims` simulations per move, subtree reuse as in the reference; finished games are restarted so the batch
    stays full (steady state, like the GPU arm).  `ply()` = one move of every game.  Falls back to the oracle's C port of
    the tree when oracle/_ref is absent."""

    def __init__(self, trees: int = 256, sims: int = SELFPLAY_SIMS, threads: int | None = None):
        import numpy as np
        import torch

        import oracle

        self.np, self.torch, self.oracle = np, torch, oracle
        self.cores = threads or os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        self.model = _default_model().eval()
        self.trees, self.sims = int(trees), int(sims)
        self.kind, self.portable = "port", None
        ref_dir = ROOT / "oracle" / "_ref"
        if list(ref_dir.glob("_liuzhou_portable_cpp*.so")):
            try:
                sys.path.insert(0, str(ref_dir))
                import _liuzhou_portable_cpp as portable

                self.portable, self.kind = portable, "reference"
            except Exception:
                self.portable = None
        states = oracle.initial_states(self.trees)
        # diversify like the GPU arm: game i advanced by a different number of uniform-random plies
        for i in range(self.trees):
            tr = oracle.random_playout(SEED, i, (120 * i) // max(1, self.trees - 1), want_trace=False)
            if not oracle.is_game_over(tr["final"]):
                for k in oracle.STATE_FIELDS:
                    states[k][i] = np.asarray(tr["final"][k])[0]
        self.tb = self._new_tree(states)
        self.positions = self.evals = 0

    def _new_tree(self, st):
        np = self.np
        if self.portable is not None:
            from types import SimpleNamespace

            objs = []
            for i in range(st["board"].shape[0]):
                objs.append(SimpleNamespace(
                    board=[[int(v) for v in row] for row in st["board"][i].reshape(6, 6)], phase=int(st["phase"][i]),
                    current_player=int(st["current_player"][i]),
                    marked_black=[(int(r), int(c)) for r, c in zip(*np.nonzero(st["marks_black"][i].reshape(6, 6)))],
                    marked_white=[(int(r), int(c)) for r, c in zip(*np.nonzero(st["marks_white"][i].reshape(6, 6)))],
                    forced_removals_done=int(st["forced_removals_done"][i]), move_count=int(st["move_count"][i]),
                    pending_marks_required=int(st["pending_marks_required"][i]),
                    pending_marks_remaining=int(st["pending_marks_remaining"][i]),
                    pending_captures_required=int(st["pending_captures_required"][i]),
                    pending_captures_remaining=int(st["pending_captures_remaining"][i]),
                    moves_since_capture=int(st["moves_since_capture"][i])))
            return self.portable.PortableTreeBatch(objs, exploration_weight=1.0, num_threads=self.cores)
        return self.oracle.TreeBatch(st, 1.0)

    def _evaluate(self, inputs, masks):
        from liuzhou_b200.net import bucket_logits_to_scalar

        np, torch = self.np, self.torch
        with torch.inference_mode():
            lp1, lp2, lpm, vl = self.model(torch.from_numpy(inputs))
            pri, _ = self.oracle.project_policy_logits_fast(lp1.numpy(), lp2.numpy(), lpm.numpy(), masks != 0)
            return pri.astype(np.float32), bucket_logits_to_scalar(vl).numpy().astype(np.float32)

    def _complete(self, pend):
        np = self.np
        n = len(pend["tree_indices"])
        if n:
            self.tb.complete_pending(*self._evaluate(pend["model_inputs"], pend["legal_masks"]))
        else:
            self.tb.complete_pending(np.zeros((0, 220), np.float32), np.zeros((0,), np.float32))
        self.evals += n

    def ply(self) -> int:
        """One move of every live game (sims simulations each); returns the positions produced."""
        np, tb = self.np, self.tb
        self._complete(tb.prepare_roots())
        for _ in range(self.sims):
            self._complete(tb.select_leaves())
        out = tb.root_outputs()
        live = out["terminal"] == 0
        n = int(live.sum())
        self.positions += n
        actions = np.where(live, out["visit_counts"].argmax(1), -1).astype(np.int32)
        tb.advance_roots([int(a) for a in actions] if self.portable is not None else actions)
        if n < self.trees:        # steady state: a session whose games have all ended starts over from fresh positions
            if n == 0:
                self.tb = self._new_tree(self.oracle.initial_states(self.trees))
        return n

    def describe(self) -> str:
        tree = "reference _liuzhou_portable_cpp tree" if self.kind == "reference" else "oracle C tree port"
        return (f"{tree} + fp32 PyTorch ChessNet on {self.cores} host threads, {self.trees} concurrent games "
                f"(network batches of up to {self.trees}), subtree reuse as in the reference")


def cpu_selfplay_baseline(budget_s: float = 20.0, trees: int = 256, sims: int = SELFPLAY_SIMS,
                          threads: int | None = None) -> dict:
    """Bounded sample of the same workload on the host cores: one continuous CpuSelfPlaySession, as many plies as start
    within the budget (at least one)."""
    sess = CpuSelfPlaySession(trees=trees, sims=sims, threads=threads)
    t0 = time.perf_counter()
    plies = 0
    while True:
        sess.ply()
        plies += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {"value": sess.positions / dt, "unit": "positions/s", "cores": sess.cores, "kind": sess.kind,
            "sims_per_sec": sess.positions * sims / dt, "network_evals_per_sec": sess.evals / dt,
            "sample": f"{trees} games x {sims} sims/move, {plies} plies = {sess.positions} positions in {dt:.1f}s, "
                      f"one continuous session; {sess.describe()}"}


def sustained_replay_ms(replay, stream, seconds: float = 1.0, warm_seconds: float = 0.6, max_reps: int = 0) -> float:
    """Average duration of `replay()` over a LONG back-to-back run (default 1 s after 0.6 s of warm-up), so that the
    clocks are the power-capped steady-state ones the real step runs at -- a 30-replay burst after an idle period runs
    ~10 % faster (measured) and would overstate the fraction of the *sustained* peak."""
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    replay()
    e0.record(stream)
    for _ in range(10):
        replay()
    e1.record(stream)
    e1.synchronize()
    per = max(1e-3, e0.elapsed_time(e1) / 10)
    warm = max(10, int(warm_seconds * 1e3 / per))
    reps = max(20, int(seconds * 1e3 / per))
    if max_reps:
        warm, reps = min(warm, max_reps), min(reps, max_reps)
    for _ in range(warm):
        replay()
    e0.record(stream)
    for _ in range(reps):
        replay()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def time_trunk_conv(net, n, stream, reps: int = 30) -> dict:
    """One trunk layer of the network = one launch of conv_tc_kernel<9,2>; both epilogue variants (conv1: bias +
    ReLU; conv2: residual + BatchNorm + ReLU, two outputs), each timed with CUDA events over graph replays."""
    import torch

    from liuzhou_b200.net import conv_bf16

    t = net.trunk._t
    if not (net.trunk is not None and net.trunk.use_tc and n % 64 == 0):
        return {"ms": float("nan"), "ms_conv1": float("nan"), "ms_conv2": float("nan"), "tflops": float("nan"),
                "ms_in_chain": float("nan"), "tflops_in_chain": float("nan"), "launches_in_chain": 0,
                "flops_per_state": 0.0, "traffic_bytes": None, "traffic_source": None}
    dev = net.device
    cl = torch.channels_last
    # post-ReLU statistics like the real activations (half zeros): tensor-core power, and with it the clock under the
    # power cap, depends on the operand data
    a = torch.relu(torch.randn((n, 128, 6, 6), device=dev, dtype=torch.bfloat16)).contiguous(memory_format=cl)
    res = torch.randn_like(a)
    o1, o2 = torch.empty_like(a), torch.empty_like(a)

    def replay_ms(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        return sustained_replay_ms(g.replay, stream, seconds=0.7, warm_seconds=0.4)

    ms1 = replay_ms(lambda: conv_bf16(a, t["wp1_0"], bias=t["bf1_0"], relu1=True, out1=o1))
    ms2 = replay_ms(lambda: conv_bf16(a, t["wp2_0"], residual=res, scale=t["s1_1"], shift=t["t1_1"], want_out2=True,
                                      out1=o1, out2=o2))
    # the same 20 launches as they run in the forward: one chain (conv1, conv2) x 10 with programmatic dependent launch
    # between the layers (a layer's prologue / weight prefetch overlaps the previous layer's epilogue)
    nb = len(net.trunk.model.blocks)

    # The 20 trunk launches as they run in the forward -- the product's own FusedTrunk.__call__ on real channel-padded
    # inputs: stem + (conv1, conv2) x 10 with programmatic dependent launch between the layers, X updated in place, three
    # activation buffers.  The stem launch (K = 64) is timed alone in the same way and subtracted, so the figure is the
    # average duration of a 3x3 128 -> 128 launch inside the chain.
    x_in = net.new_input(n)
    x_in[:, :11] = (torch.rand((n, 11, 6, 6), device=dev) > 0.6).to(torch.bfloat16)
    xo1, xo2 = torch.empty_like(a), torch.empty_like(a)
    ms_stem = replay_ms(lambda: conv_bf16(x_in, t["stem_wp"], bias=t["stem_bf"], relu1=True, scale=t["s1_0"],
                                          shift=t["t1_0"], want_out2=True, out1=xo1, out2=xo2))
    ms_trunk = replay_ms(lambda: net.trunk(x_in))
    ms_chain = (ms_trunk - ms_stem) / max(1, 2 * nb)
    flops_per_state = 2.0 * 36 * 128 * 128 * 9
    ms = 0.5 * (ms1 + ms2)
    # per-launch DRAM traffic: read from the committed ncu --set full summary of this kernel (4,096-state launch), scaled by n
    t4096, traffic_src = ncu_dram_traffic("conv_pad_kernel<9, 2>")
    traffic = None if t4096 is None else t4096 * n / 4096.0
    return {"ms": ms, "ms_conv1": ms1, "ms_conv2": ms2, "tflops": n * flops_per_state / (ms / 1e3) / 1e12,
            "ms_in_chain": ms_chain, "tflops_in_chain": n * flops_per_state / (ms_chain / 1e3) / 1e12,
            "launches_in_chain": 2 * nb, "ms_stem_launch": ms_stem, "ms_trunk": ms_trunk,
            "flops_per_state": flops_per_state, "traffic_bytes": traffic,
            "traffic_source": traffic_src}


def time_fused_trunk(net, n, stream, x_real=None) -> dict:
    """The dominant kernel of the default build: `trunk_kernel` (csrc/lz_trunk.cu) = stem + 20 residual-block convs +
    the heads' 1x1 conv in ONE persistent launch.  Timed alone with CUDA events over >= 0.7 s of back-to-back graph
    replays (power-capped steady-state clocks) on real encoded positions.  Algorithmic FLOPs per state = 2 x MACs of
    those 22 convolutions with the stem at its true 11 input channels (the kernel runs it zero-padded to 64)."""
    import torch

    if not getattr(net, "fused_trunk", False):
        return None
    dev = net.device
    x = net.new_input(n)
    if x_real is not None:
        x.copy_(x_real)
    else:
        x[:, :11] = (torch.rand((n, 11, 6, 6), device=dev) > 0.6).to(torch.bfloat16)
    for _ in range(3):
        net._trunk_heads_conv(x)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        net._trunk_heads_conv(x)
    ms = sustained_replay_ms(g.replay, stream, seconds=0.7, warm_seconds=0.4)
    nb = len(net.model.blocks)
    flops = 2.0 * 36 * 9 * 11 * 128 + 2 * nb * (2.0 * 36 * 9 * 128 * 128) + 2.0 * 36 * 128 * 128
    t, src = ncu_dram_traffic("trunk_kernel")
    return {"ms": ms, "flops_per_state": flops, "tflops": n * flops / (ms / 1e3) / 1e12, "traffic_bytes": t,
            "traffic_source": src, "launches_per_forward": 1}


def time_tree_kernels(stepper, peaks, reps: int = 20) -> dict:
    """select and expand+backup of one simulation wave, launched eagerly and timed with CUDA events on their stream
    (inside the wave graph they run back to back with the network); algorithmic bytes from the tree's own counters:
    select  = 28 B per sibling record scanned (visit 4 + info 4 + first_child 4 + prior 8 + value_sum 8) + per
              simulation 12 B root header + 32 B leaf state read + 32 B leaf state / 8 B slot / 136 B path written;
    expand  = per expanded leaf 32 B state + 880 B priors + 4 B value read, 64 B per child node written,
              12 B read + 12 B written per node on the backed-up path + 136 B path read."""
    import torch

    from liuzhou_b200.tree import encode_inputs

    m, tree = stepper.mcts, stepper.mcts.tree
    stream = torch.cuda.current_stream(stepper.device)
    torch.cuda.synchronize()
    c0 = tree.stats()
    ev = []
    for _ in range(reps):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record(stream)
        tree.select_leaves()
        e[1].record(stream)
        encode_inputs(tree.pending_states, "bf16_nhwc", out=m._wave_in)
        m._wave_forward(None)
        e[2].record(stream)
        tree.complete_pending(m._wave_pri, m._wave_val)
        e[3].record(stream)
        ev.append(e)
    torch.cuda.synchronize()
    c1 = tree.stats()
    sel_ms = sum(e[0].elapsed_time(e[1]) for e in ev) / reps
    exp_ms = sum(e[2].elapsed_time(e[3]) for e in ev) / reps
    sims = reps * tree.num_trees * tree.k
    sibs = (c1["siblings_scanned"] - c0["siblings_scanned"]) & 0xFFFFFFFF        # 32-bit wrapping device counters
    levels = (c1["levels_descended"] - c0["levels_descended"]) & 0xFFFFFFFF
    new_nodes = c1["nodes_used"] - c0["nodes_used"]
    expansions = c1["expansions"] - c0["expansions"]
    sel_bytes = sibs * 28 + sims * (12 + 32 + 32 + 8 + 136)
    exp_bytes = expansions * (32 + 880 + 4) + new_nodes * 64 + (levels + sims) * 24 + sims * 136
    sel_gbs = sel_bytes / reps / (sel_ms / 1e3) / 1e9
    exp_gbs = exp_bytes / reps / (exp_ms / 1e3) / 1e9
    # the kernel the wave actually runs: expand + backup of wave w and select (+ input encoding) of wave w + 1 fused,
    # timed in a sustained stream of [network, fused kernel] pairs
    fused_ms = None
    if m._fused_encode(m._wave_in):
        tree.select_leaves(m._wave_in)
        fe = []
        for i in range(3 * reps):
            m._wave_forward(None)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            tree.complete_and_select(m._wave_pri, m._wave_val, m._wave_in)
            b.record(stream)
            fe.append((a, b))
        m._wave_forward(None)
        tree.complete_pending(m._wave_pri, m._wave_val)
        torch.cuda.synchronize()
        fused_ms = sum(a.elapsed_time(b) for a, b in fe[reps:]) / (2 * reps)
    per_wave_bytes = (sel_bytes + exp_bytes) / reps + tree.num_trees * tree.k * 1152          # + the encoded inputs (16 of 64 channels)
    return {"bound": "hbm (latency-limited: one dependent HBM round trip per tree level, one warp per tree)",
            "expand_select_fused_ms": fused_ms,
            "expand_select_fused_gbs": None if not fused_ms else per_wave_bytes / (fused_ms / 1e3) / 1e9,
            "expand_select_fused_frac": None if not fused_ms else per_wave_bytes / (fused_ms / 1e3) / 1e9 / peaks["hbm_gbs"],
            "select_ms": sel_ms, "expand_backup_ms": exp_ms, "select_gbs": sel_gbs, "expand_backup_gbs": exp_gbs,
            "peak_gbs": peaks["hbm_gbs"], "select_frac": sel_gbs / peaks["hbm_gbs"],
            "expand_backup_frac": exp_gbs / peaks["hbm_gbs"],
            "bytes_per_simulation": (sel_bytes + exp_bytes) / max(1, sims), "avg_depth": levels / max(1, sims),
            "avg_siblings_per_level": sibs / max(1, levels), "children_per_expansion": new_nodes / max(1, expansions),
            "ncu": "profiles/r02_tree_heads_ncu_full.csv (DRAM bytes, occupancy, issue utilisation); timeline: tools/trace_tree.py"}


def run_selfplay(args, world, rank, local_rank):
    import torch

    from liuzhou_b200 import _lib
    from liuzhou_b200.engine import BYTES_PER_POSITION, SelfPlayStepper
    from liuzhou_b200.net import InferenceNet

    dev = torch.device("cuda", local_rank)
    peaks, peak_kind = measured_peaks()
    games, sims, k = args.games, args.sims, args.leaves_per_wave
    model = _default_model()
    if world > 1:   # weights come from rank 0 over NCCL (replaces the reference's torch.save / torch.load hand-off)
        import torch.distributed as dist

        model = model.to(dev)
        for t in list(model.parameters()) + list(model.buffers()):
            dist.broadcast(t.data, src=0)
    net = InferenceNet(model, dev)
    torch.manual_seed(SEED * 10007 + (rank + 1) * 9973)          # per-rank seed rule of v1/train.py:795,998
    stepper = SelfPlayStepper(net, games, simulations=sims, leaves_per_wave=k, seed=SEED, device=dev,
                              reuse_subtree=bool(args.tree_reuse))
    stepper.diversify(seed=SEED + rank)
    stream = torch.cuda.current_stream(dev)

    # N > 1: this ply's trajectory rows (all five tensors of the reference format) return to the trainer rank over NCCL
    # as fixed-size compact rows (liuzhou_b200/compact.py: 336 B instead of 2,692 B per position, lossless; static
    # shapes, so nothing on the path synchronises with the host).  Compaction + gather are queued on a side stream and
    # overlap the next ply's search; the ring keeps 4 plies, and before ply p the main stream waits for the gather of
    # ply p-3, so a slot is never overwritten while in flight.
    side = torch.cuda.Stream(dev) if world > 1 else None
    gather_done = []

    def step():
        if world > 1 and len(gather_done) >= 3:
            stream.wait_event(gather_done[-3])
        stepper.step()
        if world > 1:
            from liuzhou_b200.compact import compact_rows_fixed
            from liuzhou_b200.dist import gather_rows_fixed
            from liuzhou_b200.trajectory_buffer import TensorSelfPlayBatch

            side.wait_stream(stream)
            with torch.cuda.stream(side):
                planes, legal, policy, _sign = stepper.trajectory_block()
                nan = torch.full((games,), float("nan"), device=dev)
                gather_rows_fixed(compact_rows_fixed(TensorSelfPlayBatch(planes, legal, policy, nan, nan)), dst=0)
                ev = torch.cuda.Event()
                ev.record(side)
                gather_done.append(ev)
                del gather_done[:-4]

    for _ in range(args.warmup):
        step()
    barrier_sync(world)
    launches0 = _lib.launch_count()
    evals0 = stepper.mcts.evals
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    if world > 1:
        stream.wait_stream(side)          # the last ply's gather is inside the timed region
    e1.record(stream)
    e1.synchronize()
    barrier_sync(world)
    clocks = sampler.stop() if rank == 0 else {}
    if args.dump_outputs and rank == 0:
        # the last timed ply: its trajectory rows (reference format), the positions after the move (finished games
        # refilled), the ply counters and the running outcome counts
        from liuzhou_b200 import native
        from liuzhou_b200._lib import STATE_FIELDS

        planes, legal, policy, sign = stepper.trajectory_block()
        state = {f"state_{k}": t for k, t in zip(STATE_FIELDS, native.unpack_states(stepper.states))}
        dump_outputs(args.dump_outputs, {"trajectory_planes": planes, "trajectory_legal_mask": legal,
                                         "trajectory_policy": policy, "trajectory_sign": sign, **state,
                                         "plies": stepper.plies}, {"outcomes": stepper.outcomes})
    # graph replays re-launch the captured kernels: our kernels inside the root / wave graphs were counted at capture
    waves = stepper.mcts.waves
    launches = (_lib.launch_count() - launches0) + args.steps * (waves * stepper.mcts.wave_graph_launches
                                                                 + stepper.mcts.root_graph_launches
                                                                 + stepper.mcts.search_extra_launches)
    rank_ms = all_ranks(e0.elapsed_time(e1), world)
    elapsed_ms = max(rank_ms)                                         # max over ranks, device-timed
    positions = sum_over_ranks(float(games * args.steps), world)
    value = positions / (elapsed_ms / 1e3)
    evals = stepper.mcts.evals - evals0

    if args.profile_only:
        if rank == 0:
            print(json.dumps({"metric": "selfplay_positions_per_sec", "value": value, "unit": "positions/s",
                              "ms_per_step": elapsed_ms / args.steps, "gpu_launches": int(launches),
                              "note": "--profile-only: device-timed steps only"}), flush=True)
        raise SystemExit(0)
    # dominant kernel group: the network forward (PyTorch / cuDNN, bf16 tensor cores) at the wave batch size,
    # timed alone with CUDA events on its stream; the tree kernels are the remainder of the wave.
    slots = games * k
    x = net.new_input(slots)
    # real positions as input: tensor-core power (hence the clock under the power cap) depends on the data -- an
    # all-zero input runs the same forward ~15 % faster and would not describe the forward inside a wave
    from liuzhou_b200.tree import encode_inputs as _encode_inputs

    _encode_inputs(stepper.states.repeat(k, 1) if k > 1 else stepper.states, "bf16_nhwc", out=x)
    g = torch.cuda.CUDAGraph()
    for _ in range(3):
        net._forward_eager(x)
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        net._forward_eager(x)
    # sustained (power-capped) clocks: 1 s of forward replays, then -- without a pause -- 200 wave replays (one ply's
    # worth; more would overrun the node arena)
    fwd_ms = sustained_replay_ms(g.replay, stream, seconds=1.0, warm_seconds=0.6)
    stepper.mcts._first_graph.replay()           # the wave graph is [network, expand + next select]: it needs a select first
    wave_ms = sustained_replay_ms(stepper.mcts._wave_graph.replay, stream, max_reps=100)
    stepper.mcts._last_graph.replay()            # ... and the last network + expand leaves nothing pending
    tflops = slots * net.flops_per_state / (fwd_ms / 1e3) / 1e12
    tree_roof = time_tree_kernels(stepper, peaks)
    tree_stats = stepper.mcts.tree.stats()
    fused = time_fused_trunk(net, slots, stream, x_real=x)
    conv = time_trunk_conv(net, slots, stream)

    # e2e: the PUBLIC ENTRY end to end -- one full self_play_v1_gpu(search_backend="tree") iteration per rank from a HOST
    # model (weights H2D + BatchNorm folding inside the timed region), all games from the initial
    # position to their end with the reference's wave semantics (no refill), value-target finalisation, and the finished
    # TensorSelfPlayBatch copied to pinned host memory (D2H).  N > 1: every rank plays its own iteration (weights
    # broadcast from rank 0 first) and the compact trajectory gather to rank 0 is inside the timed region too.
    from liuzhou_b200.self_play import self_play_v1_gpu

    del stepper
    torch.cuda.empty_cache()
    host_model = _default_model()
    h2d = int(sum(t.numel() * t.element_size() for t in list(host_model.parameters()) + list(host_model.buffers())))
    # warm-up (untimed), as for the device-timed steps: the actor's long-lived objects -- inference wrapper, tree arenas,
    # the CUDA graphs of a full-size wave -- are built by a 3-ply run of the same entry; a self-play worker keeps them
    # across iterations the same way (run_self_play_worker: one InferenceNet + one engine cache per worker)
    e2e_net = InferenceNet(_default_model(), dev)
    engines: dict = {}
    kw_entry = dict(num_games=games, mcts_simulations=sims, temperature_init=1.0, temperature_final=0.1,
                    temperature_threshold=10, exploration_weight=1.0, device=str(dev), add_dirichlet_noise=True,
                    concurrent_games=games, search_backend="tree", leaves_per_wave=k,
                    tree_reuse=bool(args.tree_reuse), engine_cache=engines)
    self_play_v1_gpu(e2e_net, max_game_plies=3, **kw_entry)
    # the actor's pinned staging area for finished trajectories is long-lived too (self_play_storage keeps its staging
    # slots the same way): page-locking 1.4 GB costs ~0.4 s and is not part of an iteration.  Sized for 160 positions
    # per game; a longer iteration falls back to allocating inside the timed region.
    pin_rows = games * 160 * (world if rank == 0 else 0)
    pin_shapes = (((11, 6, 6), torch.float32), ((220,), torch.bool), ((220,), torch.float32), ((), torch.float32),
                  ((), torch.float32))
    pinned = [torch.empty((pin_rows,) + shp, dtype=dt, pin_memory=True) for shp, dt in pin_shapes] if pin_rows else None
    torch.manual_seed(SEED * 10007 + (rank + 1) * 9973 + 17)
    barrier_sync(world)
    marks = {}
    t0 = time.perf_counter()
    if world > 1:
        import torch.distributed as dist
        from liuzhou_b200 import dist as lzdist

        dev_model = host_model.to(dev)
        lzdist.broadcast_model(dev_model, src=0)
        e2e_net.load_state_dict(dev_model.state_dict())
    else:
        e2e_net.load_state_dict(host_model.state_dict())           # this iteration's weights: host -> device, refolded
    torch.cuda.synchronize()
    marks["weights_s"] = time.perf_counter() - t0
    fb, fs = self_play_v1_gpu(e2e_net, **kw_entry)
    torch.cuda.synchronize()
    marks["self_play_s"] = time.perf_counter() - t0 - marks["weights_s"]
    gathered_positions = None
    if world > 1:
        merged = lzdist.gather_trajectories_compact(fb, dst=0)
        out_b = merged if rank == 0 else None
        gathered_positions = merged.num_samples if rank == 0 else 0
    else:
        out_b = fb
    d2h = 0
    if out_b is not None:
        fields = (out_b.state_tensors, out_b.legal_masks, out_b.policy_targets, out_b.value_targets,
                  out_b.soft_value_targets)
        if pinned is not None and fields[0].shape[0] <= pin_rows:
            host = [p[: t.shape[0]] for p, t in zip(pinned, fields)]
        else:
            host = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in fields]
        for dst, src in zip(host, fields):
            dst.copy_(src, non_blocking=True)
        d2h = int(sum(h.numel() * h.element_size() for h in host))
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    marks["handoff_s"] = e2e_s - marks["weights_s"] - marks["self_play_s"]
    e2e_elapsed = max_over_ranks(e2e_s, world)
    e2e_positions = sum_over_ranks(float(fb.num_samples), world)
    e2e_value = e2e_positions / e2e_elapsed
    full_line = {"positions": int(e2e_positions), "seconds": e2e_elapsed, "plies_to_last_game_end": None,
                 "avg_game_length": fs.avg_game_length, "black_wins": fs.black_wins, "white_wins": fs.white_wins,
                 "draws": fs.draws, "gathered_positions_on_rank0": gathered_positions,
                 "stages_rank0_s": {k_: round(v_, 4) for k_, v_ in marks.items()},
                 "what": "one full self_play_v1_gpu(search_backend='tree') iteration per rank on a warmed-up actor, wall clock "
                         "incl. weight H2D + refolding, trajectory finalisation"
                         + (", NCCL weight broadcast + compact trajectory gather to rank 0" if world > 1 else "")
                         + " and the D2H copy of the finished batch to pinned memory"}
    del fb, out_b
    net = e2e_net

    # the same workload on the reference's production backend (root-only PUCT through the drop-in v0_core ops): one
    # warm-up + one timed full self_play_v1_gpu iteration; reported next to the tree-search headline (N = 1 only)
    root_line = None
    if world == 1 and not args.no_root_line:
        from liuzhou_b200.self_play import self_play_v1_gpu

        def root_iteration(seed):
            torch.manual_seed(seed)
            return self_play_v1_gpu(net, num_games=games, mcts_simulations=sims, temperature_init=1.0,
                                    temperature_final=0.1, temperature_threshold=10, exploration_weight=1.0,
                                    device=str(dev), add_dirichlet_noise=True, concurrent_games=games,
                                    search_backend="root")

        torch.cuda.empty_cache()
        root_iteration(SEED)
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record(stream)
        rb, _rs = root_iteration(SEED + 1)
        r1.record(stream)
        r1.synchronize()
        root_line = {"value": rb.num_samples / (r0.elapsed_time(r1) / 1e3), "unit": "positions/s",
                     "positions": rb.num_samples, "seconds": r0.elapsed_time(r1) / 1e3,
                     "what": "one full self_play_v1_gpu iteration, search_backend=root (reference production path), "
                             "same games / sims / net; see bench.py --search root"}

    # the v1 REFERENCE itself on this GPU (its python + its v0_core CUDA + its PyTorch network), same games / sims:
    # the denominator of north_star's ">= 100x the v1 reference per GPU" (N = 1 only; own process, after ours has finished)
    ref_gpu = None
    if world == 1 and args.ref_gpu:
        torch.cuda.empty_cache()
        ref_gpu = reference_gpu_line(games, sims, local_rank)
    legacy = legacy_cpu_line() if (world == 1 and rank == 0 and args.legacy_cpu) else None

    if rank != 0:
        return None
    peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
    cpu = cpu_selfplay_baseline(budget_s=args.cpu_budget, sims=sims)
    return {
        "metric": "selfplay_positions_per_sec", "value": value, "unit": "positions/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps,
        "ms_per_step_by_rank": [m / args.steps for m in rank_ms],
        "root_puct_backend": root_line, "tree_backend_full_iteration": full_line, "reference_gpu": ref_gpu,
        "config1_legacy_cpu": legacy,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "mcts_sims_per_sec": value * sims, "network_evals_per_sec": evals * world / (elapsed_ms / 1e3),
        "config": {"workload": "v1 wave-batched MCTS self-play (BASELINE configs[2])", "games_per_gpu": games,
                   "sims_per_move": sims, "search": "full tree on device (select/expand/backup kernels)",
                   "leaves_per_wave": k,
                   "subtree_reuse": bool(args.tree_reuse) and "advance_roots after every move (portable_cpp_self_play.py:170): "
                                    "200 NEW simulations per move on top of the inherited subtree, arena compacted per ply",
                   "net": "ChessNet 128ch x 10 blocks, random init, seed 20260314; all 22 convolutions of a forward run in ONE "
                          "persistent tcgen05 kernel of ours (trunk_kernel), no cuDNN on the path",
                   "step": "one ply of every game; finished games refilled; batch pre-diversified by 0..120 random plies",
                   "dirichlet_noise": True, "temperature": "1.0 -> 0.1 at ply 10", "exploration_weight": 1.0,
                   "l2": "working set per step (node arena > 1 GB) exceeds the 126 MB L2",
                   "comparisons": {
                       "public_entry_full_iteration_positions_per_sec": e2e_value,
                       "public_entry_vs_stepper": e2e_value / value if value else None,
                       "ours_root_puct_backend_positions_per_sec": None if not root_line else root_line["value"],
                       "reference_gpu_root_puct_positions_per_sec": None if not ref_gpu else ref_gpu.get("value"),
                       "ours_root_vs_reference_gpu": (root_line["value"] / ref_gpu["value"])
                       if (root_line and ref_gpu and ref_gpu.get("value")) else None,
                       "ours_tree_positions_vs_reference_gpu_root_positions (different searches: 200 vs ~15 evals per position)": (value / ref_gpu["value"])
                       if (ref_gpu and ref_gpu.get("value")) else None,
                       "config1_legacy_cpu_positions_per_sec": None if not legacy else legacy.get("value")}},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "positions/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": 1, "step": "one full self_play_v1_gpu(search_backend='tree') iteration per rank (public entry): "
                                    f"{int(e2e_positions)} positions in {e2e_elapsed:.2f} s", "detail": full_line},
        "gpu_launches": int(launches),
        # dominant kernel: our tcgen05 implicit-GEMM convolution (20 of the 22 launches per forward are this 3x3
        # 128->128 instance); achieved = algorithmic FLOPs of one launch / its CUDA-event duration in a graph replay
        # (average launch duration = the 20-launch trunk chain / 20, the way the launches run inside the step; a launch
        # replayed alone, without the PDL overlap with its neighbours, is reported next to it)
        "roofline": ({"bound": "tensor", "achieved": fused["tflops"], "peak": peak, "unit": "TFLOP/s",
                      "frac": fused["tflops"] / peak, "traffic": fused["traffic_bytes"],
                      "peak_kind": peak_kind + " (sustained bf16, cuBLAS)",
                      "kernel": "trunk_kernel (csrc/lz_trunk.cu: stem + 20 residual-block 3x3 convs + heads 1x1 conv in ONE "
                                "persistent launch; bf16 tcgen05.mma cta_group::2, activations resident in shared memory / "
                                "TMEM, taps via shifted UMMA descriptors, fp32 residual stream in TMEM)",
                      "kernel_ms": fused["ms"], "units_per_launch": slots, "flops_per_unit": fused["flops_per_state"],
                      "launches_per_forward": 1,
                      "traffic_source": f"ncu --set full dram__bytes_read+write per launch, {fused['traffic_source']}",
                      "forward_ms": fwd_ms, "forward_tflops": tflops, "forward_frac_of_peak": tflops / peak,
                      "wave_ms": wave_ms, "share_of_step": fused["ms"] * (waves + 1) / (elapsed_ms / args.steps),
                      "per_layer_kernels (LZB_TRUNK_IMPL=0)": {
                          "kernel": "conv_pad_kernel<9,2> (csrc/lz_conv.cu), one launch per convolution",
                          "ms_in_chain": conv["ms_in_chain"], "tflops_in_chain": conv["tflops_in_chain"],
                          "frac_in_chain": conv["tflops_in_chain"] / peak, "ms_trunk_21_launches": conv.get("ms_trunk")}}
                     if fused else
                     {"bound": "tensor", "achieved": conv["tflops_in_chain"], "peak": peak, "unit": "TFLOP/s",
                      "frac": conv["tflops_in_chain"] / peak, "traffic": conv["traffic_bytes"],
                      "kernel_ms_in_chain": conv["ms_in_chain"], "achieved_launch_alone": conv["tflops"],
                      "frac_launch_alone": conv["tflops"] / peak,
                      "peak_kind": peak_kind + " (sustained bf16, cuBLAS)",
                      "kernel": "conv_pad_kernel<9,2> (csrc/lz_conv.cu: 3x3 128->128 conv, bf16 tcgen05.mma cta_group::2, "
                                "padded boards in shared memory, fused bias/residual/BN/ReLU epilogue)",
                      "kernel_ms": conv["ms"], "kernel_ms_conv1_epilogue": conv["ms_conv1"],
                      "kernel_ms_conv2_epilogue": conv["ms_conv2"], "units_per_launch": slots,
                      "flops_per_unit": conv["flops_per_state"], "launches_per_forward": 20,
                      "traffic_source": f"ncu --set full dram__bytes_read+write per launch, {conv['traffic_source']}",
                      "forward_ms": fwd_ms, "forward_tflops": tflops, "forward_frac_of_peak": tflops / peak,
                      "wave_ms": wave_ms,
                      "share_of_step": 20 * conv["ms_in_chain"] * (waves + 1) / (elapsed_ms / args.steps)}),
        "tree": tree_stats,
        "tree_roofline": tree_roof,
        "cpu_baseline": cpu,
    }


def run_selfplay_root(args, world, rank, local_rank):
    """The reference's PRODUCTION search (`--search_backend cuda_root`: root-only PUCT, v1/python/mcts_gpu.py:1249-1457)
    through our drop-in entry: one step = one full `self_play_v1_gpu` iteration (all games played to the end), which
    is what v1/train.py runs per worker and what the reference's published H20 numbers measure (BASELINE.md section 1)."""
    import torch

    from liuzhou_b200 import _lib
    from liuzhou_b200.net import InferenceNet
    from liuzhou_b200.self_play import self_play_v1_gpu

    dev = torch.device("cuda", local_rank)
    peaks, peak_kind = measured_peaks()
    games, sims = args.games, args.sims
    model = _default_model()
    if world > 1:
        import torch.distributed as dist

        model = model.to(dev)
        for t in list(model.parameters()) + list(model.buffers()):
            dist.broadcast(t.data, src=0)
    net = InferenceNet(model, dev)
    stream = torch.cuda.current_stream(dev)

    def iteration(seed):
        torch.manual_seed(seed * 10007 + (rank + 1) * 9973)
        return self_play_v1_gpu(net, num_games=games, mcts_simulations=sims, temperature_init=1.0, temperature_final=0.1,
                                temperature_threshold=10, exploration_weight=1.0, device=str(dev),
                                add_dirichlet_noise=True, soft_value_k=2.0, max_game_plies=512, sample_moves=True,
                                concurrent_games=games, search_backend="root")

    for w in range(max(1, min(args.warmup, 1))):
        iteration(SEED + w)
    barrier_sync(world)
    launches0 = _lib.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = args.steps
    positions = 0
    last = None
    e0.record(stream)
    for it in range(steps):
        batch, stats = iteration(SEED + 100 + it)
        positions += batch.num_samples
        last = (batch, stats)
    e1.record(stream)
    e1.synchronize()
    barrier_sync(world)
    clocks = sampler.stop() if rank == 0 else {}
    elapsed_ms = max_over_ranks(e0.elapsed_time(e1), world)
    launches = _lib.launch_count() - launches0
    all_positions = sum_over_ranks(float(positions), world)
    value = all_positions / (elapsed_ms / 1e3)
    # e2e: the same iteration with the resulting trajectory batch (reference format, 2,692 B/position) read to the host
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    batch, stats = iteration(SEED + 200)
    host = batch.to("cpu")
    e2e_s = time.perf_counter() - t0
    e2e_value = sum_over_ranks(float(host.num_samples), world) / max_over_ranks(e2e_s, world)
    conv = time_trunk_conv(net, 4096, stream)
    ref_gpu = None
    if world == 1 and args.ref_gpu:
        del net
        torch.cuda.empty_cache()
        ref_gpu = reference_gpu_line(games, sims, local_rank)
    if rank != 0:
        return None
    peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
    st = last[1]
    cpu = cpu_selfplay_baseline(budget_s=args.cpu_budget, sims=sims)
    return {
        "metric": "selfplay_positions_per_sec", "value": value, "unit": "positions/s", "n_gpus": world, "steps": steps,
        "warmup": 1, "ms_per_step": elapsed_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic", "mcts_sims_per_sec": value * sims,
        "config": {"workload": "v1 wave-batched self-play, root-PUCT search (the reference's production backend; BASELINE "
                               "configs[2] with search_backend=cuda_root)", "games_per_gpu": games, "sims_per_move": sims,
                   "search": "root-only PUCT: 1 + #legal-children network evaluations per position, root_puct kernel",
                   "step": "one full self_play_v1_gpu iteration (every game played to its end, trajectory batch built)",
                   "net": "ChessNet 128ch x 10 blocks, random init, seed 20260314", "dirichlet_noise": True,
                   "temperature": "1.0 -> 0.1 at ply 10",
                   "l2": "activations of a child batch (>= 100 MB per tensor) exceed the 126 MB L2",
                   "published_reference": "4,995.8 positions/s on 1 x H20 at sims=1024, 64 concurrent games "
                                          "(v1/Design.md:1528; other hardware / config, so vs_baseline stays null)",
                   "comparisons": {
                       "reference_gpu_root_puct_positions_per_sec": None if not ref_gpu else ref_gpu.get("value"),
                       "ours_vs_reference_gpu": (value / ref_gpu["value"]) if (ref_gpu and ref_gpu.get("value")) else None,
                       "ours_e2e_vs_reference_gpu_e2e": (e2e_value / ref_gpu["e2e"]["value"])
                       if (ref_gpu and ref_gpu.get("value")) else None}},
        "reference_gpu": ref_gpu,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "positions/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": int(host.nbytes())},
        "gpu_launches": int(launches),
        "selfplay_stats": {"games": st.num_games, "positions": st.num_positions, "avg_game_length": st.avg_game_length,
                           "black_wins": st.black_wins, "white_wins": st.white_wins, "draws": st.draws},
        # (average launch duration = the 20-launch trunk chain / 20, the way the launches run inside the step; a launch
        # replayed alone, without the PDL overlap with its neighbours, is reported next to it)
        "roofline": {"bound": "tensor", "achieved": conv["tflops_in_chain"], "peak": peak, "unit": "TFLOP/s",
                     "frac": conv["tflops_in_chain"] / peak, "traffic": conv["traffic_bytes"],
                     "kernel_ms_in_chain": conv["ms_in_chain"], "achieved_launch_alone": conv["tflops"],
                     "frac_launch_alone": conv["tflops"] / peak,
                     "peak_kind": peak_kind + " (sustained bf16, cuBLAS)",
                     "kernel": "conv_tc_kernel<9,2> (csrc/lz_conv.cu)", "kernel_ms": conv["ms"], "units_per_launch": 4096,
                     "flops_per_unit": conv["flops_per_state"]},
        "cpu_baseline": cpu,
    }


def run_config4(args, world, rank, local_rank):
    """BASELINE configs[3]: self-play sharded by game over the GPUs of one box -- 4,096 games per GPU (32,768 on 8) x 800
    sims/move through `liuzhou_b200.dist.self_play_sharded`: NCCL weight broadcast from rank 0, per-rank seeds
    (iteration_seed * 10007 + (rank + 1) * 9973), one full `self_play_v1_gpu(search_backend="tree")` iteration per rank,
    the compact trajectory gather to rank 0 and the stats all-reduce -- ALL inside the timed region (one step = one
    training iteration's self-play stage, v1/train.py:129-135,932-1171).  e2e adds the D2H copy of the merged batch."""
    import torch

    from liuzhou_b200 import _lib
    from liuzhou_b200 import dist as lzdist

    dev = torch.device("cuda", local_rank)
    games, sims = args.games, args.sims
    total = games * world
    model = _default_model()
    kw = dict(mcts_simulations=sims, temperature_init=1.0, temperature_final=0.1, temperature_threshold=10,
              exploration_weight=1.0, add_dirichlet_noise=True, soft_value_k=2.0, max_game_plies=512,
              sample_moves=True, concurrent_games=games, search_backend="tree")
    # warm-up: CUDA context, NCCL communicator, allocator (a tiny sharded iteration)
    lzdist.self_play_sharded(_default_model(), 64 * world, iteration_seed=1, device=dev,
                             **{**kw, "mcts_simulations": 8, "concurrent_games": 64})
    # rank 0's long-lived pinned staging area for the merged batch (160 positions per game; longer iterations fall back
    # to allocating inside the timed region)
    pin_rows = total * 160 if rank == 0 else 0
    pinned = None
    if pin_rows:
        try:
            pinned = [torch.empty((pin_rows,) + shp, dtype=dt, pin_memory=True)
                      for shp, dt in (((11, 6, 6), torch.float32), ((220,), torch.bool), ((220,), torch.float32),
                                      ((), torch.float32), ((), torch.float32))]
        except RuntimeError:
            pinned = None
    barrier_sync(world)
    launches0 = _lib.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    t0 = time.perf_counter()
    timings: dict = {}
    merged, summary = lzdist.self_play_sharded(model, total, iteration_seed=SEED, device=dev, timings=timings, **kw)
    torch.cuda.synchronize()
    t_dev = time.perf_counter() - t0
    d2h = 0
    if merged is not None:
        fields = (merged.state_tensors, merged.legal_masks, merged.policy_targets, merged.value_targets,
                  merged.soft_value_targets)
        if pinned is not None and fields[0].shape[0] <= pin_rows:
            host = [p[: t.shape[0]] for p, t in zip(pinned, fields)]
        else:
            host = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in fields]
        for dst, src in zip(host, fields):
            dst.copy_(src, non_blocking=True)
        d2h = int(sum(h.numel() * h.element_size() for h in host))
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    barrier_sync(world)
    clocks = sampler.stop() if rank == 0 else {}
    play_ms = all_ranks(timings["self_play_s"] * 1e3, world)
    elapsed = max_over_ranks(t_dev, world)
    e2e_elapsed = max_over_ranks(t_e2e, world)
    handoff_ms = max_over_ranks(timings["handoff_s"] * 1e3, world)
    bcast_ms = max_over_ranks(timings["broadcast_s"] * 1e3, world)
    launches = _lib.launch_count() - launches0
    if rank != 0:
        return None
    tot = [summary["num_games"], summary["num_positions"], summary["black_wins"], summary["white_wins"], summary["draws"]]
    positions = tot[1]
    value = positions / elapsed
    h2d = int(sum(t.numel() * t.element_size() for t in list(model.parameters()) + list(model.buffers())))
    return {
        "metric": "selfplay_positions_per_sec", "value": value, "unit": "positions/s", "n_gpus": world, "steps": 1,
        "warmup": 1, "ms_per_step": elapsed * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic", "mcts_sims_per_sec": value * sims,
        "config": {"workload": "self-play sharded by game with NCCL weight broadcast + trajectory gather (BASELINE "
                               "configs[3])", "games_total": total, "games_per_gpu": games, "sims_per_move": sims,
                   "search": "full tree on device", "step": "one training iteration's self-play stage, end to end",
                   "net": "ChessNet 128ch x 10 blocks, random init, seed 20260314",
                   "l2": "working set per step (node arena > 1 GB) exceeds the 126 MB L2"},
        "clocks": clocks,
        "e2e": {"value": positions / e2e_elapsed, "unit": "positions/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches),
        "iteration": {"positions": int(positions), "games": int(tot[0]), "black_wins": int(tot[2]),
                      "white_wins": int(tot[3]), "draws": int(tot[4]), "seconds": elapsed,
                      "self_play_ms_by_rank": play_ms, "weight_broadcast_ms": bcast_ms,
                      "handoff_ms (compact gather + stats all-reduce)": handoff_ms,
                      "merged_positions_on_rank0": None if merged is None else int(merged.num_samples)},
    }


def reference_cpu_entry_line(games: int = 64, sims: int = SELFPLAY_SIMS, plies: int = 1, timeout_s: float = 240.0):
    """The reference's OWN CPU full-tree self-play entry, unmodified (`self_play_v1_portable_cpp`,
    v1/python/portable_cpp_self_play.py:26, via oracle/ref_runner.py portable): a bounded run next to the CPU arm, which
    drives the same compiled tree from a leaner loop of ours and is the faster -- hence the more conservative -- baseline."""
    if not (ROOT / "oracle" / "_ref" / "pysrc").is_dir():
        return {"unavailable": "oracle/_ref/pysrc not present on this box"}
    import subprocess
    try:
        res = subprocess.run([sys.executable, str(ROOT / "oracle" / "ref_runner.py"), "portable", "--games", str(games),
                              "--sims", str(sims), "--max-plies", str(plies), "--warmup-games", "8"],
                             capture_output=True, text=True, timeout=timeout_s)
        r = json.loads(res.stdout.strip().splitlines()[-1])
    except Exception as exc:  # pragma: no cover
        return {"unavailable": f"ref_runner portable failed: {exc!r}"[:200]}
    if "positions_per_sec" not in r:
        return r
    return {"value": r["positions_per_sec"], "unit": "positions/s", "sims_per_sec": r["sims_per_sec"], "cores": r["cores"],
            "positions": r["positions"], "seconds": r["seconds"],
            "what": f"{r['what']}: {games} games x {sims} sims, {plies} ply per game"}


def run_reference_selfplay(args):
    """--impl reference: the reference's CPU implementation of the path on all host cores, ONE continuous session (no
    restarts between steps); a step = one move of every game of the session, its duration is measured.  The session is
    a bounded sample of the workload: `--ref-trees` concurrent games (default 256, so the CPU network sees batches of
    256), shrunk once -- before the timed region -- if the first ply shows that K + W plies would not fit ~4 minutes."""
    trees = int(args.ref_trees)
    sess = CpuSelfPlaySession(trees=trees, sims=args.sims)
    t0 = time.perf_counter()
    sess.ply()
    first = time.perf_counter() - t0
    plies_needed = args.warmup + args.steps
    budget = float(args.ref_budget)
    if first * plies_needed > budget and trees > 32:
        trees = max(32, int(trees * budget / (first * plies_needed)) // 32 * 32)
        sess = CpuSelfPlaySession(trees=trees, sims=args.sims)
        sess.ply()
    for _ in range(max(0, args.warmup - 1)):
        sess.ply()
    p0, e0 = sess.positions, sess.evals
    step_s = []
    for _ in range(args.steps):
        t = time.perf_counter()
        sess.ply()
        step_s.append(time.perf_counter() - t)
    dt = sum(step_s)
    positions = sess.positions - p0
    value = positions / dt
    cpu = {"value": value, "unit": "positions/s", "cores": sess.cores, "kind": sess.kind,
           "sims_per_sec": value * args.sims, "network_evals_per_sec": (sess.evals - e0) / dt,
           "sample": f"{trees} games x {args.sims} sims/move, {args.steps} timed plies = {positions} positions in "
                     f"{dt:.1f}s after {args.warmup} warm-up plies, one continuous session; {sess.describe()}"}
    return {
        "impl": "reference", "metric": "selfplay_positions_per_sec", "value": value, "unit": "positions/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "mcts_sims_per_sec": value * args.sims,
        "config": {"workload": "v1 wave-batched MCTS self-play (BASELINE configs[2])", "sims_per_move": args.sims,
                   "games": trees, "same_config": False,
                   "search": "reference CPU tree (portable C++) + fp32 network on host cores",
                   "step": "one move of every game of one continuous session (measured, not a fixed budget)"},
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": "positions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "reference_cpu_entry": reference_cpu_entry_line(sims=args.sims) if args.ref_entry else None,
    }


# ----------------------------------------------------------------------------------------------------
# workload: config 5 -- checkpoint eval vs the random agent (2,000 games, 64 sims) + 4-checkpoint round robin
# ----------------------------------------------------------------------------------------------------
def run_eval(args, world, rank, local_rank):
    import torch

    from liuzhou_b200 import _lib
    from liuzhou_b200.evaluate import play_match, round_robin_tournament
    from liuzhou_b200.net import ChessNet, InferenceNet

    dev = torch.device("cuda", local_rank)
    games, sims = args.eval_games, args.eval_sims
    nets = []
    for sd in (1, 2, 3, 4):           # SURVEY 8d-5: four random-init checkpoints, seeds 1-4
        torch.manual_seed(sd)
        nets.append(InferenceNet(ChessNet(), dev))
    play_match(nets[0], None, num_games=128, mcts_simulations=sims, device=dev, seed=0)     # warm-up: graph capture
    barrier_sync(world)
    launches0 = _lib.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    stream = torch.cuda.current_stream(dev)
    e0.record(stream)
    stats = play_match(nets[0], None, num_games=games, mcts_simulations=sims, temperature=0.0, device=dev,
                       seed=SEED + rank)
    e1.record(stream)
    rr = round_robin_tournament(nets, games_per_match=args.eval_rr_games, mcts_simulations=sims, temperature=1.0,
                                sample_moves=True, device=dev, seed=SEED + rank)
    e2.record(stream)
    e2.synchronize()
    barrier_sync(world)
    clocks = sampler.stop() if rank == 0 else {}
    ms_eval = max_over_ranks(e0.elapsed_time(e1), world)
    ms_rr = max_over_ranks(e1.elapsed_time(e2), world)
    total_games = sum_over_ranks(float(stats.total_games), world)
    plies = sum_over_ranks(float(stats.plies), world)
    if rank != 0:
        return None
    return {
        "metric": "eval_games_per_sec", "value": total_games / (ms_eval / 1e3), "unit": "games/s", "n_gpus": world,
        "steps": 1, "warmup": 1, "ms_per_step": ms_eval, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "checkpoint eval vs random agent + 4-checkpoint round robin (BASELINE configs[4])",
                   "games_per_gpu": stats.total_games, "sims_per_move": sims, "temperature": 0.0,
                   "round_robin": f"4 random-init checkpoints (seeds 1-4), {args.eval_rr_games} games per pairing, T=1 sampled"},
        "clocks": clocks, "positions_per_sec": plies / (ms_eval / 1e3),
        "eval": {"wins": stats.wins, "losses": stats.losses, "draws": stats.draws, "plies": stats.plies,
                 "searched_positions": stats.searches, "color_breakdown": stats.color_breakdown},
        "round_robin": {"ms": ms_rr, "standings": [{k: r[k] for k in ("name", "match_points", "game_wins", "game_losses",
                                                                        "game_draws")} for r in rr["standings"]]},
        "gpu_launches": int(_lib.launch_count() - launches0),
    }


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=SELFPLAY_GAMES)
    ap.add_argument("--sims", type=int, default=SELFPLAY_SIMS)
    ap.add_argument("--leaves-per-wave", type=int, default=1)
    ap.add_argument("--tree-reuse", type=int, default=1,
                    help="1: the played child's subtree is kept between moves (advance_roots, as the reference's "
                         "portable self-play does); 0: every search starts from a bare root")
    ap.add_argument("--no-root-line", action="store_true", help="skip the extra root-PUCT iteration in the default line")
    ap.add_argument("--search", choices=["tree", "root"], default="tree",
                    help="tree: device-resident full tree (north_star, default); root: the reference's root-PUCT backend")
    ap.add_argument("--ref-entry", type=int, default=1,
                    help="--impl reference: also time the reference's own self_play_v1_portable_cpp entry (64 games x 1 ply)")
    ap.add_argument("--profile-only", action="store_true",
                    help="for ncu launch lists: only the device-timed steps (no e2e iteration, no reference / CPU legs)")
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--ref-trees", type=int, default=256, help="--impl reference: concurrent games of the CPU session")
    ap.add_argument("--ref-budget", type=float, default=240.0, help="--impl reference: target wall time of the whole run (s)")
    ap.add_argument("--ref-gpu", type=int, default=1,
                    help="1: also time the UNMODIFIED v1 reference (its python + its v0_core CUDA) on the same GPU (N = 1)")
    ap.add_argument("--legacy-cpu", type=int, default=1, help="1: also time BASELINE configs[0] (legacy src/ self-play, CPU)")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 5); config4 and eval time one whole run, so only 1 is accepted there")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=["playout", "selfplay", "eval", "config4"], default="selfplay")
    ap.add_argument("--eval-games", type=int, default=2000)
    ap.add_argument("--eval-sims", type=int, default=64)
    ap.add_argument("--eval-rr-games", type=int, default=256)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (default self-play "
                         "workload; rank 0's games)")
    args = ap.parse_args()
    if args.workload in ("config4", "eval") and args.impl == "ours":
        if args.steps not in (None, 1):
            ap.error(f"--workload {args.workload} times one whole run: --steps must be 1")
        args.steps = 1
    args.steps = 5 if args.steps is None else args.steps
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl, args.workload, args.search) != ("ours", "selfplay", "tree"):
        ap.error("--dump-outputs is implemented for the default workload (--impl ours --workload selfplay --search tree)")
    args.warmup = max(3, args.warmup) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return 0
        fn = run_reference_selfplay if args.workload == "selfplay" else run_reference_playout
        print(json.dumps(fn(args)), flush=True)
        return 0

    world, rank, local_rank = dist_setup(args.gpus)
    if args.workload == "config4" and args.sims == SELFPLAY_SIMS:
        args.sims = 800
    fn = {"selfplay": run_selfplay_root if args.search == "root" else run_selfplay, "playout": run_playout,
          "eval": run_eval, "config4": run_config4}[args.workload]
    line = fn(args, world, rank, local_rank)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
