"""SelfPlayActor checks that need no GPU: argument refusals and the memory arithmetic."""
import pytest

from liuzhou_b200 import actor
from liuzhou_b200.compact import FIXED_ROW_WORDS


def test_arena_and_output_sizes():
    assert actor.ROW_BYTES == FIXED_ROW_WORDS * 8 == 336
    # one fixed row + an int8 sign + an int16 action per (slot, ply), an int32 row count per slot
    assert actor.arena_bytes(4096, 512) == 4096 * 512 * 339 + 4096 * 4
    assert 0.70e9 < actor.arena_bytes(4096, 512) < 0.72e9
    assert actor.arena_bytes(1, 1) == 339 + 4
    # per output row: the fixed row, an int16 action and (at most one game per row) a 64-byte record
    assert actor.output_bytes(1000) == 1000 * (336 + 2 + 64)


@pytest.mark.parametrize("kw", [dict(num_games=0), dict(num_games=-3), dict(max_game_plies=0),
                                dict(max_game_plies=-1), dict(mcts_simulations=0), dict(leaves_per_wave=0),
                                dict(max_game_plies=64, output_capacity=63)])
def test_constructor_refuses_bad_sizes(kw):
    args = dict(num_games=8, device="cuda", mcts_simulations=4)
    args.update(kw)
    with pytest.raises(ValueError):
        actor.SelfPlayActor(None, args.pop("num_games"), **args)


def test_constructor_refuses_cpu_device():
    with pytest.raises(RuntimeError, match="CUDA"):
        actor.SelfPlayActor(None, 8, device="cpu")
