"""SelfPlayActor (liuzhou_b200/actor.py, csrc/lz_actor.cu) on the GPU: without refill it reproduces the wave entry
bit for bit; with refill every emitted game replays on the CPU oracle with the stored targets; the record kernel
writes exactly compact_rows_fixed's words; emission is deterministic, overflow is loud, and a ply never waits for the
host."""
import ctypes
import math

import numpy as np
import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
KW = dict(mcts_simulations=16, temperature_init=1.0, temperature_final=0.1, temperature_threshold=10,
          exploration_weight=1.0, add_dirichlet_noise=True, soft_value_k=2.0, sample_moves=True)


def _net(seed=0):
    from liuzhou_b200.net import ChessNet, InferenceNet

    torch.manual_seed(seed)
    return InferenceNet(ChessNet(), DEV)


def _actor(net, g, **kw):
    from liuzhou_b200.actor import SelfPlayActor

    args = dict(KW)
    args.update(kw)
    return SelfPlayActor(net, g, device=DEV, **args)


def _replay_check(games, max_plies, k=2.0):
    """Every game of a drain, replayed from its action trace on the oracle."""
    b = games.batch
    planes, legal = b.state_tensors.cpu().numpy(), b.legal_masks.cpu().numpy()
    policy = b.policy_targets.cpu().numpy()
    actions = games.actions.cpu().numpy()
    lengths, offsets = games.length.cpu().tolist(), games.row_offset.cpu().tolist()
    results, softs = games.result.cpu().numpy(), games.soft_value.cpu().numpy()
    assert sum(lengths) == b.num_samples == games.rows.shape[0]
    for i, (length, r0) in enumerate(zip(lengths, offsets)):
        st = oracle.initial_states(1)
        signs = []
        stuck = False
        for j in range(length):
            row = r0 + j
            assert not oracle.is_game_over(st), (i, j)
            assert np.array_equal(planes[row], oracle.states_to_model_input(st)[0]), (i, j)
            assert np.array_equal(legal[row], oracle.encode_actions_fast(st)[0][0]), (i, j)
            assert (policy[row][~legal[row]] == 0).all()
            signs.append(int(st["current_player"][0]))
            a = int(actions[row])
            scalar_legal = oracle.legal_actions(st)[0]
            if a < 0:                                            # no legal action: the side to move loses
                assert j == length - 1 and len(scalar_legal) == 0
                assert (policy[row] == 0).all()
                stuck = True
                break
            assert a in scalar_legal, (i, j, a)
            assert abs(float(policy[row].sum(dtype=np.float64)) - 1.0) <= 1e-6
            st = oracle.apply_move_scalar(st, a)
        if stuck:
            expect = -signs[-1]
        elif oracle.is_game_over(st):
            expect = oracle.winner(st)
        else:
            assert length == max_plies, (i, length)
            expect = 0
        assert results[i] == expect, (i, results[i], expect)
        board = st["board"][0]
        d = torch.tensor([int((board == 1).sum()) - int((board == -1).sum())], dtype=torch.int64, device=DEV)
        s_ref = torch.tanh(d.to(torch.float32) / 18.0 * float(k))
        assert int(games.piece_delta[i]) == int(d)
        assert softs[i] == float(s_ref), i
        sg = torch.tensor(signs, dtype=torch.float32, device=DEV)
        assert torch.equal(b.value_targets[r0:r0 + length], sg * float(expect))
        assert torch.equal(b.soft_value_targets[r0:r0 + length], sg * s_ref)


def _ply_major(games, g):
    """Row permutation that puts the drained rows into the wave loop's ply-major, slot-ascending order."""
    keys = []
    for slot, length, r0 in zip(games.slot.tolist(), games.length.tolist(), games.row_offset.tolist()):
        keys += [(j * g + slot, r0 + j) for j in range(length)]
    keys.sort()
    return torch.tensor([r for _, r in keys], dtype=torch.int64, device=DEV)


@pytest.mark.parametrize("g", [128, 100, 300])          # 300: two emit blocks, games ending in the same ply in both
def test_refill_off_equals_wave_entry(g):
    from liuzhou_b200.self_play import self_play_v1_gpu

    net = _net(3)
    torch.manual_seed(1234)
    ref, ref_stats = self_play_v1_gpu(net, num_games=g, concurrent_games=g, device=DEV, search_backend="tree",
                                      opening_random_moves=4, **KW)
    torch.manual_seed(1234)
    act = _actor(net, g, opening_random_moves=4, output_capacity=g * 512)   # the whole wave in one drain
    act.finish()
    while not act.idle:
        act.step(plies=16)
    games = act.drain()
    assert games.stats.num_games == g and sorted(games.slot.tolist()) == list(range(g))
    perm = _ply_major(games, g)
    for f in ("state_tensors", "legal_masks", "policy_targets", "value_targets", "soft_value_targets"):
        assert torch.equal(getattr(games.batch, f).index_select(0, perm), getattr(ref, f)), f
    s = games.stats
    assert (s.black_wins, s.white_wins, s.draws) == (ref_stats.black_wins, ref_stats.white_wins, ref_stats.draws)
    assert s.num_positions == ref_stats.num_positions
    assert abs(s.avg_game_length - ref_stats.avg_game_length) < 1e-4
    assert s.piece_delta_buckets == ref_stats.piece_delta_buckets
    # per-game lengths and results in slot order
    order = torch.argsort(games.slot)
    res = games.result[order]
    assert [int((res > 0).sum()), int((res < 0).sum()), int((res == 0).sum())] == [s.black_wins, s.white_wins, s.draws]


@pytest.mark.parametrize("g", [64, 300])
def test_refill_on_replays_on_oracle(g):
    max_plies = 40
    torch.manual_seed(7)
    act = _actor(_net(5), g, mcts_simulations=8, max_game_plies=max_plies, opening_random_moves=2)
    serials, positions, lengths, checked_refill = [], 0, 0, False
    for _ in range(4):
        act.step(plies=25)
        games = act.drain()
        assert games.stats.num_games == games.serial.numel()          # none before ply 40 of the first games
        _replay_check(games, max_plies)
        serials += games.serial.tolist()
        positions += games.batch.num_samples
        lengths += int(games.length.sum())
        checked_refill |= bool((games.serial >= g).any())
        assert (games.finish_step >= 0).all() and (games.finish_step < act.steps).all()
    assert checked_refill and len(serials) > g
    assert len(set(serials)) == len(serials) and sorted(serials) == list(range(len(serials)))
    assert positions == lengths


def test_record_kernel_matches_compact_rows_fixed():
    from liuzhou_b200 import native
    from liuzhou_b200._lib import lib, ptr, stream_ptr
    from liuzhou_b200.compact import FIXED_ROW_WORDS, compact_rows_fixed
    from liuzhou_b200.trajectory_buffer import TensorSelfPlayBatch
    from liuzhou_b200.tree import encode_inputs

    n = 1024
    pb_states = []
    for i, steps in enumerate((0, 5, 20, 40, 70, 100, 130, 160)):
        pb = native.PlayoutBatch(n // 8, seed=99, device=DEV, game_offset=i * 1000)
        if steps:
            pb.run(max_steps=steps)
        pb_states.append(pb.packed)
    states = torch.cat(pb_states).contiguous()
    legal = native.mask_words_to_bool(native.legal_masks(states, scalar_semantics=False)[0])
    gen = torch.Generator(device=DEV).manual_seed(5)
    pol = torch.rand((n, 220), device=DEV, generator=gen) * legal
    pol = pol / pol.sum(1, keepdim=True).clamp_min(1e-30)
    pol[3, (~legal[3]).nonzero()[0, 0]] = 0.25                   # mass off the legal set: not representable
    pol[5] = 0.0                                                   # an all-zero row
    nan = torch.full((n,), float("nan"), device=DEV)
    ref = compact_rows_fixed(TensorSelfPlayBatch(encode_inputs(states, "f32_nchw"), legal, pol, nan, nan.clone()))
    arena = torch.full((n, FIXED_ROW_WORDS), 0x0123456789, dtype=torch.int64, device=DEV)
    signs = torch.zeros((n,), dtype=torch.int8, device=DEV)
    acts = torch.zeros((n,), dtype=torch.int16, device=DEV)
    nrows = torch.zeros((n,), dtype=torch.int32, device=DEV)
    ctl = torch.zeros((48,), dtype=torch.int64, device=DEV)
    active = torch.ones((n,), dtype=torch.uint8, device=DEV)
    chosen = torch.arange(n, dtype=torch.int64, device=DEV) % 220 - 1
    rc = lib().lzb_actor_record(ptr(states), ptr(active), ptr(pol), ptr(chosen), ctypes.c_int64(n), ctypes.c_int32(1),
                                ptr(nrows), ptr(arena), ptr(signs), ptr(acts), ptr(ctl), stream_ptr(DEV))
    assert rc == 0
    assert torch.equal(arena, ref)
    assert int(arena[3, 41]) == 1 and int((arena[:, 41] != 0).sum()) == 1
    white = (states[:, 0] >> 39) & 1
    assert torch.equal(signs, (1 - 2 * white).to(torch.int8))
    assert torch.equal(acts, chosen.to(torch.int16)) and bool((nrows == 1).all()) and int(ctl.abs().sum()) == 0
    # a full arena is refused loudly, not overwritten
    rc = lib().lzb_actor_record(ptr(states), ptr(active), ptr(pol), ptr(chosen), ctypes.c_int64(n), ctypes.c_int32(1),
                                ptr(nrows), ptr(arena), ptr(signs), ptr(acts), ptr(ctl), stream_ptr(DEV))
    assert rc == 0 and torch.equal(arena, ref) and int(ctl[3]) == 2


def _run(seed, g=64, steps=45, **kw):
    torch.manual_seed(seed)
    act = _actor(_net(5), g, mcts_simulations=8, max_game_plies=40, **kw)
    act.step(plies=steps)
    return act


@pytest.mark.parametrize("g", [64, 300])
def test_emission_is_deterministic_and_overflow_is_loud(g):
    runs = [_run(11, g=g).drain() for _ in range(2)]
    a, b = runs
    assert a.stats.num_games > 0
    for f in ("rows", "actions", "serial", "slot", "length", "row_offset", "finish_step", "piece_delta", "result",
              "soft_value"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    # too small an output: the kernel writes nothing past the end, the drain raises
    torch.manual_seed(11)
    act = _actor(_net(5), g, mcts_simulations=8, max_game_plies=40, output_capacity=40)
    guard = 16
    rows = torch.full((40 + guard, 42), 0x5A5A5A5A5A5A5A5A, dtype=torch.int64, device=DEV)
    acts = torch.full((40 + guard,), 0x5A5A, dtype=torch.int16, device=DEV)
    recs = torch.full((40 + guard, 8), 0x5A5A5A5A5A5A5A5A, dtype=torch.int64, device=DEV)
    act._out_rows, act._out_actions, act._records = rows[:40], acts[:40], recs[:40]
    act.step(plies=45)
    with pytest.raises(RuntimeError, match="overflow"):
        act.drain()
    assert bool((rows[40:] == 0x5A5A5A5A5A5A5A5A).all()) and bool((acts[40:] == 0x5A5A).all())
    assert bool((recs[40:] == 0x5A5A5A5A5A5A5A5A).all())
    # the overflowed output was discarded: the actor goes on with an empty output
    assert act.drain().stats.num_games == 0


def test_step_does_not_synchronise_while_refilling():
    act = _run(3, steps=36, opening_random_moves=4)               # the first search captures the graphs
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        act.step(plies=6)              # every game reaches 40 plies and refills: plies 0, 1 of the random opening
    finally:
        torch.cuda.set_sync_debug_mode(0)
    games = act.drain()
    assert games.stats.num_games >= 64 and bool((games.finish_step >= 36).any())
    _replay_check(games, 40)


def test_new_weights_mid_run():
    from liuzhou_b200 import native
    from liuzhou_b200.net import ChessNet, InferenceNet
    from liuzhou_b200.tree import encode_inputs

    act = _run(21, steps=10)
    act.drain()
    torch.manual_seed(77)
    model2 = ChessNet()
    act.load_state_dict(model2.state_dict())
    fresh = InferenceNet(model2, DEV)
    pb = native.PlayoutBatch(128, seed=3, device=DEV)
    pb.run(max_steps=30)
    states = pb.packed
    outs = []
    for net in (act.net, fresh):
        x = net.new_input(128)
        encode_inputs(states, "bf16_nhwc", out=x)
        pri, val = net.forward_priors(x, states)
        outs.append((pri.clone(), val.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    act.step(plies=40)
    games = act.drain()
    assert games.stats.num_games > 0 and math.isfinite(games.stats.avg_game_length)
    _replay_check(games, 40)
