"""SelfPlayActor against SelfPlayStepper, alternated in one process, and the actor's two bookkeeping kernels alone.

    python tools/bench_actor.py [--games 4096] [--sims 200] [--plies 6] [--rounds 3] [--kernel-plies 200]

1. ms per ply of ``SelfPlayStepper.step()`` and ``SelfPlayActor.step()`` (refilling, subtree reuse on, default net,
   same search settings), both diversified to a mid-game steady state, in alternating blocks of ``--plies`` plies;
   device-synchronised wall clock per block.
2. ``lzb_actor_record`` and ``lzb_actor_emit`` alone with CUDA events over ``--kernel-plies`` launches each, on the
   actor's own buffers after its plies: record writes every slot's row; emit finishes every 100th slot with a game of
   100 rows per launch (about the steady-state rate of games of ~100 plies), timed with the two small resets it needs,
   which are also timed alone.
Prints the card name and power limit with the numbers.
"""
import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from liuzhou_b200 import native  # noqa: E402
from liuzhou_b200.actor import SelfPlayActor  # noqa: E402
from liuzhou_b200.engine import SelfPlayStepper  # noqa: E402
from liuzhou_b200.net import ChessNet, InferenceNet  # noqa: E402


def card() -> dict:
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "unknown"
    return info


def timed(fn, n: int) -> float:
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n * 1e3


def kernel_ms(fn, n: int) -> float:
    fn()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(n):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / n


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=200)
    ap.add_argument("--plies", type=int, default=6)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--kernel-plies", type=int, default=200)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.manual_seed(20260314)
    net = InferenceNet(ChessNet(), dev)
    stepper = SelfPlayStepper(net, a.games, simulations=a.sims, device=dev, reuse_subtree=True)
    stepper.diversify()
    actor = SelfPlayActor(net, a.games, device=dev, mcts_simulations=a.sims, output_capacity=256 * a.games)
    actor.states, actor.plies = stepper.states.clone(), stepper.plies.clone()   # the same mid-game steady state
    stepper.step()                     # warm-up: graph capture of both engines
    actor.step()
    times = {"stepper": [], "actor": []}
    for _ in range(a.rounds):
        times["stepper"].append(timed(stepper.step, a.plies))
        times["actor"].append(timed(actor.step, a.plies))
    games = actor.drain()

    # the two kernels alone, on the actor's buffers: record every slot, emit ~1 % of them per launch
    g = a.games
    states = actor.states.contiguous()
    policy = torch.rand((g, 220), device=dev)
    chosen = torch.zeros((g,), dtype=torch.int64, device=dev)
    finished = torch.zeros((g,), dtype=torch.bool, device=dev)
    finished[:: 100] = True
    res = torch.zeros((g,), dtype=torch.float32, device=dev)
    legal = native.mask_words_to_bool(native.legal_masks(states, scalar_semantics=False)[0])
    policy = policy * legal
    n_rec = min(a.kernel_plies, actor.max_game_plies - 2)
    actor._nrows.zero_()                # each launch records the next row of every slot
    rec = kernel_ms(lambda: actor._record(states, actor._all, policy, chosen), n_rec)
    actor._nrows.fill_(100)

    def emit():
        actor._emit(finished, res, res, states)
        actor._nrows.fill_(100)
        actor._ctl[:2].zero_()

    em = kernel_ms(emit, a.kernel_plies)
    base = kernel_ms(lambda: (actor._nrows.fill_(100), actor._ctl[:2].zero_()), a.kernel_plies)
    emitted_bytes = int(finished.sum()) * 100 * 336
    print(json.dumps({
        "card": card(), "games": g, "sims": a.sims, "plies_per_block": a.plies,
        "stepper_ms_per_ply": [round(t, 2) for t in times["stepper"]],
        "actor_ms_per_ply": [round(t, 2) for t in times["actor"]],
        "stepper_median": round(statistics.median(times["stepper"]), 2),
        "actor_median": round(statistics.median(times["actor"]), 2),
        "actor_games_drained": games.stats.num_games, "actor_positions_drained": games.stats.num_positions,
        "record_us": round(rec * 1e3, 2), "emit_plus_resets_us": round(em * 1e3, 2),
        "resets_alone_us": round(base * 1e3, 2), "emit_bytes_per_launch": emitted_bytes,
    }, indent=1))


if __name__ == "__main__":
    main()
