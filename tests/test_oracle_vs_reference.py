"""Pin the CPU oracle (oracle/) against the reference's OWN binaries (oracle/_ref, built by oracle/build_ref.py from a
checkout of the reference).  CPU only.  Without oracle/_ref a test compares against what the reference's binaries
computed when tests/golden/make_golden.py ran them (tests/golden/*.npz: smaller samples of the same comparisons, checked
by the same functions as tests/test_oracle_golden.py).

Samplers and seeds follow the reference's tests:
  tests/v0/cuda/test_fast_legal_mask_cuda.py (seed 0xF00DCAFE, 10,000 uniformly random states, aux_dim=1)
  tests/v0/cuda/test_fast_apply_moves_cuda.py (seed 0xA11CEB0B, synthetic (state, action) pairs)
  tests/v0/test_actions.py (random legal playouts; we filter nothing because the oracle's scalar
  generator, like the reference's, returns [] on game-over states)
  tests/v1/test_portable_cpp_mcts.py:203-243 (visit counts / values identical)
"""
import numpy as np
import pytest

import oracle
from tests import test_oracle_golden as stored
from tests._util import (STATE_FIELDS, concat_states, dict_to_state, golden_states, load_golden, load_ref,
                         random_apply_batch, random_mask_states, sparse_random_states, state_obj, states_equal, to_torch)

REF = load_ref()
needs_ref = pytest.mark.skipif(REF is None, reason="oracle/_ref not built (run `python oracle/build_ref.py`); no stored "
                                                   "reference output covers this comparison")


def _torch():
    import torch

    return torch


def _ref_encode(v0_core, st, dims=(36, 144, 36, 4)):
    t = to_torch(st)
    mask, meta = v0_core.encode_actions_fast(*t[:10], *dims)
    return mask.numpy(), meta.numpy()


@pytest.mark.parametrize("sampler,seed", [(random_mask_states, 0xF00DCAFE), (sparse_random_states, 0x5EED)])
@pytest.mark.parametrize("aux", [1, 4])
def test_encode_actions_fast_matches_reference(sampler, seed, aux):
    if REF is None:          # stored: 2,048 states of the first sampler, then 1,024 of the second
        z = load_golden("encode_actions")
        rows = slice(0, 2048) if sampler is random_mask_states else slice(2048, None)
        mask, meta = oracle.encode_actions_fast({k: v[rows] for k, v in golden_states(z).items()}, 36, 144, 36, aux)
        assert np.array_equal(mask, np.unpackbits(z[f"mask_aux{aux}"][rows], axis=1)[:, :216 + aux].astype(bool))
        assert np.array_equal(meta, z[f"meta_aux{aux}"][rows].astype(np.int32))
        return
    v0_core, _ = REF
    st = sampler(10_000, seed)
    dims = (36, 144, 36, aux)
    ref_mask, ref_meta = _ref_encode(v0_core, st, dims)
    mask, meta = oracle.encode_actions_fast(st, *dims)
    assert np.array_equal(mask, ref_mask)
    assert np.array_equal(meta, ref_meta)


def _collect_playout_states(num_games, seed, every=1):
    states = []
    for g in range(num_games):
        trace = oracle.random_playout(seed, g, 512, want_trace=True)["trace"]
        st = oracle.initial_states(1)
        for ply, a in enumerate(trace):
            if ply % every == 0:
                states.append(st)
            st = oracle.apply_move_scalar(st, int(a))
        states.append(st)  # terminal state too
    return concat_states(states)


def test_scalar_engine_matches_reference_on_playouts():
    """legal list, next state, game-over and winner == reference scalar engine (via the portable module,
    which is built from v0/src/{game,rules,moves}/*.cpp) on every state of 40 random playouts."""
    if REF is None:
        return stored.test_scalar_playouts_golden()
    _, portable = REF
    checked = 0
    for g in range(40):
        trace = oracle.random_playout(0x7777, g, 512, want_trace=True)["trace"]
        st = oracle.initial_states(1)
        for a in list(trace) + [None]:
            info = portable.inspect_state(state_obj(st))
            idx, _codes = oracle.legal_actions(st)
            assert list(info["legal_action_indices"]) == idx
            assert bool(info["game_over"]) == oracle.is_game_over(st)
            assert int(info["winner"]) == oracle.winner(st)
            assert np.array_equal(np.asarray(info["model_input"], np.float32), oracle.states_to_model_input(st)[0])
            if a is None:
                break
            # every legal child, not only the one played
            for cand in idx:
                ref_next = dict_to_state(portable.apply_action(state_obj(st), int(cand)))
                assert states_equal(oracle.apply_move_scalar(st, int(cand)), ref_next)
                checked += 1
            st = oracle.apply_move_scalar(st, int(a))
        assert oracle.is_game_over(st) or not oracle.legal_actions(st)[0]
    assert checked > 20_000


def test_tensor_ops_match_reference_on_playouts():
    """encode_actions_fast + batch_apply_moves (all children) == v0_core CPU on reachable states."""
    if REF is None:          # stored: every legal child of the states of 6 playouts
        z = load_golden("apply_moves")
        mask, meta = oracle.encode_actions_fast(golden_states(z, "in_"))
        rows, cols = np.nonzero(mask)
        assert np.array_equal(rows, z["parents"]) and np.array_equal(meta[rows, cols], z["codes"])
        return stored.test_apply_moves_golden()
    v0_core, _ = REF
    torch = _torch()
    st = _collect_playout_states(60, 0xBEEF)
    n = st["board"].shape[0]
    ref_mask, ref_meta = _ref_encode(v0_core, st)
    mask, meta = oracle.encode_actions_fast(st)
    assert np.array_equal(mask, ref_mask) and np.array_equal(meta, ref_meta)
    # mask == scalar legal list on non-terminal states (SURVEY.md section 4 parity contract)
    for i in range(0, n, 7):
        if not oracle.is_game_over(st, i):
            assert list(np.nonzero(mask[i])[0]) == oracle.legal_actions(st, i)[0]
    rows, cols = np.nonzero(mask)
    codes = meta[rows, cols]
    parents = rows.astype(np.int64)
    ref_out = v0_core.batch_apply_moves(*to_torch(st), torch.from_numpy(codes), torch.from_numpy(parents))
    out, applied = oracle.batch_apply_moves(st, codes, parents, return_applied=True)
    assert applied.all()
    for k, ref_t in zip(STATE_FIELDS, ref_out):
        assert np.array_equal(np.asarray(out[k]).reshape(ref_t.shape), ref_t.numpy()), k
    assert codes.shape[0] > 50_000


@needs_ref
def test_apply_moves_reference_sampler():
    """The reference's synthetic (state, action) sampler: rows the CPU path accepts must match bit-exactly;
    rows it rejects (TORCH_CHECK) must be flagged `applied == False` by the oracle's CUDA-semantics port."""
    v0_core, _ = REF
    torch = _torch()
    st, codes, parents = random_apply_batch(3000, 0xA11CEB0B)
    out, applied = oracle.batch_apply_moves(st, codes, parents, return_applied=True)
    n_ok = 0
    for i in range(codes.shape[0]):
        one = {k: v[i:i + 1] for k, v in st.items()}
        try:
            ref = v0_core.batch_apply_moves(*to_torch(one), torch.from_numpy(codes[i:i + 1]),
                                            torch.zeros(1, dtype=torch.int64))
        except RuntimeError:
            assert not applied[i]
            continue
        assert applied[i]
        n_ok += 1
        for k, ref_t in zip(STATE_FIELDS, ref):
            assert np.array_equal(np.asarray(out[k][i]).reshape(ref_t.shape[1:]), ref_t.numpy()[0]), (i, k)
    assert n_ok > 1500


def test_states_to_model_input_matches_reference():
    if REF is None:
        z = load_golden("composites")
        mi = oracle.states_to_model_input(golden_states(z))
        assert np.array_equal(np.packbits(mi.astype(np.uint8)), z["model_input"])
        return
    v0_core, _ = REF
    st = random_mask_states(2000, 11)
    t = to_torch(st)
    ref = v0_core.states_to_model_input(*t[:5]).numpy()
    assert np.array_equal(oracle.states_to_model_input(st), ref)


def test_root_puct_matches_reference():
    if REF is None:
        return stored.test_root_puct_golden()
    v0_core, _ = REF
    torch = _torch()
    rng = np.random.default_rng(5)
    for (r, m, sims, c) in [(64, 40, 200, 1.0), (16, 7, 64, 1.5), (8, 220, 800, 1.0), (4, 1, 16, 1.0)]:
        valid = rng.random((r, m)) < 0.8
        valid[:, 0] = True
        pri = rng.random((r, m)).astype(np.float32) * valid
        pri = (pri / pri.sum(1, keepdims=True)).astype(np.float32)
        leaf = (rng.random((r, m)).astype(np.float32) * 2 - 1) * valid
        # quantised leaf values produce exact score ties -> exercises the lowest-index tie-break
        leaf[: r // 2] = np.round(leaf[: r // 2] * 4) / 4
        pri[: r // 4] = (valid[: r // 4] / valid[: r // 4].sum(1, keepdims=True)).astype(np.float32)
        ref_v, ref_w, ref_rv = v0_core.root_puct_allocate_visits(
            torch.from_numpy(pri), torch.from_numpy(leaf), torch.from_numpy(valid), sims, c)
        v, w, rv = oracle.root_puct_allocate_visits(pri, leaf, valid, sims, c)
        assert np.array_equal(v, ref_v.numpy())
        assert np.array_equal(w, ref_w.numpy())
        np.testing.assert_allclose(rv, ref_rv.numpy(), rtol=1e-5, atol=1e-6)


def _search_inputs(n_games=8, seed=3):
    st = _collect_playout_states(n_games, seed, every=3)
    rng = np.random.default_rng(seed)
    mask, meta = oracle.encode_actions_fast(st)
    probs = (rng.random(mask.shape).astype(np.float32) + 0.01) * mask
    probs = (probs / np.maximum(probs.sum(1, keepdims=True), 1e-8)).astype(np.float32)
    return st, mask, meta, probs, rng


def test_root_pack_and_finalize_match_reference():
    if REF is None:          # the stored composites: root pack, finalize, model input, projection, self-play step
        return stored.test_composites_golden()
    v0_core, _ = REF
    torch = _torch()
    st, mask, meta, probs, rng = _search_inputs()
    mask[::17] = False  # rows without legal actions -> terminal roots
    ref = v0_core.root_pack_sparse_actions(torch.from_numpy(mask), torch.from_numpy(probs), torch.from_numpy(meta))
    got = oracle.root_pack_sparse_actions(mask, probs, meta)
    for i, (g, r) in enumerate(zip(got, ref)):
        if i == 5:
            np.testing.assert_allclose(g, r.numpy(), rtol=1e-6, atol=1e-7)
        else:
            assert np.array_equal(g, r.numpy()), i
    (_tm, roots, _cnt, valid_mask, legal_idx, priors, code_mat, _flat, _ca, _pa) = got
    leaf = (rng.random(priors.shape).astype(np.float32) * 2 - 1) * valid_mask
    visits, value_sum, _ = oracle.root_puct_allocate_visits(priors, leaf, valid_mask, 128, 1.0)
    temps = np.where(np.arange(roots.size) % 2 == 0, 1.0, 0.5).astype(np.float32)
    ref = v0_core.root_finalize_from_visits(
        torch.from_numpy(legal_idx), torch.from_numpy(code_mat), torch.from_numpy(valid_mask),
        torch.from_numpy(visits), torch.from_numpy(value_sum), torch.from_numpy(roots),
        mask.shape[0], 220, torch.from_numpy(temps), False)
    got = oracle.root_finalize_from_visits(legal_idx, code_mat, valid_mask, visits, value_sum, roots,
                                           mask.shape[0], 220, temps)
    np.testing.assert_allclose(got[0], ref[0].numpy(), rtol=1e-5, atol=1e-7)   # policy (fp32 pow)
    assert np.array_equal(got[1], ref[1].numpy())
    assert np.array_equal(got[2], ref[2].numpy())
    assert np.array_equal(got[3], ref[3].numpy())
    np.testing.assert_allclose(got[4], ref[4].numpy(), rtol=1e-5, atol=1e-6)


@needs_ref
def test_root_sparse_writeback_matches_reference():
    """module.cpp:365-439: the scatter of an external legal policy + picks back to dense rows (exact: products and
    single adds only)."""
    v0_core, _ = REF
    torch = _torch()
    st, mask, meta, probs, rng = _search_inputs()
    mask[::13] = False
    (_tm, roots, cnt, valid_mask, legal_idx, priors, code_mat, _flat, _ca, _pa) = oracle.root_pack_sparse_actions(
        mask, probs, meta)
    policy = (rng.random(priors.shape).astype(np.float32) + 0.05)          # NOT masked: the op applies valid_mask itself
    picks = (rng.integers(0, 1 << 30, roots.size) % cnt).astype(np.int64)
    ref = v0_core.root_sparse_writeback(torch.from_numpy(legal_idx), torch.from_numpy(code_mat),
                                        torch.from_numpy(valid_mask), torch.from_numpy(policy), torch.from_numpy(picks),
                                        torch.from_numpy(roots), mask.shape[0], 220)
    got = oracle.root_sparse_writeback(legal_idx, code_mat, valid_mask, policy, picks, roots, mask.shape[0], 220)
    for i, (g, r) in enumerate(zip(got, ref)):
        assert np.array_equal(g, r.numpy()), i


def test_project_policy_matches_reference():
    if REF is None:
        z = load_golden("composites")
        p, _l = oracle.project_policy_logits_fast(z["head0"], z["head1"], z["head2"], z["mask"])
        np.testing.assert_allclose(p, z["proj_probs"], rtol=1e-5, atol=1e-7)
        assert np.array_equal(np.isfinite(_l), np.isfinite(z["proj_logits"]))
        fin = np.isfinite(_l)
        np.testing.assert_allclose(_l[fin], z["proj_logits"][fin], rtol=1e-6, atol=1e-6)
        return
    v0_core, _ = REF
    torch = _torch()
    st, mask, _meta, _probs, rng = _search_inputs(4, 9)
    n = mask.shape[0]
    heads = [torch.log_softmax(torch.from_numpy(rng.standard_normal((n, 36)).astype(np.float32)), 1) for _ in range(3)]
    mask[::13] = False
    ref_p, ref_l = v0_core.project_policy_logits_fast(*heads, torch.from_numpy(mask), 36, 144, 36, 4)
    p, l = oracle.project_policy_logits_fast(*(h.numpy() for h in heads), mask)
    np.testing.assert_allclose(p, ref_p.numpy(), rtol=1e-5, atol=1e-7)
    assert np.array_equal(np.isfinite(l), np.isfinite(ref_l.numpy()))
    fin = np.isfinite(l)
    np.testing.assert_allclose(l[fin], ref_l.numpy()[fin], rtol=1e-6, atol=1e-6)


def test_self_play_step_and_finalize_match_reference():
    if REF is None:          # stored: the self-play step (finalize_trajectory_inplace was not stored)
        return stored.test_composites_golden()
    v0_core, _ = REF
    torch = _torch()
    st = _collect_playout_states(12, 21, every=1)
    n = st["board"].shape[0]
    rng = np.random.default_rng(2)
    mask, meta = oracle.encode_actions_fast(st)
    # late-game rows so that win / draw / max-ply finalisation paths fire
    plies = st["move_count"].copy()
    done = np.zeros((n,), bool)
    done[::11] = True
    active = np.nonzero(~done)[0].astype(np.int64)
    terminal = ~mask[active].any(1)
    codes = np.full((active.size, 4), -1, np.int32)
    valid = np.zeros((active.size,), bool)
    for j, g in enumerate(active):
        idx = np.nonzero(mask[g])[0]
        if idx.size and rng.random() > 0.03:
            codes[j] = meta[g, rng.choice(idx)]
            valid[j] = True
    t_state = [t.clone() for t in to_torch(st)]
    t_plies, t_done = torch.from_numpy(plies.copy()), torch.from_numpy(done.copy())
    ref = v0_core.self_play_step_inplace(*t_state, t_plies, t_done, torch.from_numpy(active), torch.from_numpy(codes),
                                         torch.from_numpy(terminal), torch.from_numpy(valid), 130, 2.0)
    o_state = {k: np.array(v, copy=True) for k, v in st.items()}
    o_plies, o_done = plies.copy(), done.copy()
    got = oracle.self_play_step_inplace(o_state, o_plies, o_done, active, codes, terminal, valid, 130, 2.0)
    assert np.array_equal(got[0], ref[0].numpy())
    assert np.array_equal(got[1], ref[1].numpy())
    np.testing.assert_allclose(got[2], ref[2].numpy(), rtol=1e-6, atol=1e-7)
    assert got[0].size > 10
    for k, t in zip(STATE_FIELDS, t_state):
        assert np.array_equal(np.asarray(o_state[k]).reshape(t.shape), t.numpy()), k
    assert np.array_equal(o_plies, t_plies.numpy()) and np.array_equal(o_done, t_done.numpy())

    # finalize_trajectory_inplace on a synthetic step-index matrix
    g_count, t_max = 16, 9
    counts = rng.integers(0, t_max + 1, (g_count,)).astype(np.int64)
    sim = np.full((g_count, t_max), -1, np.int64)
    total = int(counts.sum())
    perm = rng.permutation(total)
    k = 0
    for g in range(g_count):
        sim[g, :counts[g]] = perm[k:k + counts[g]]
        k += counts[g]
    signs = rng.choice([-1, 1], total).astype(np.int8)
    slots = rng.permutation(g_count)[:10].astype(np.int64)
    res = rng.choice([-1.0, 0.0, 1.0], slots.size).astype(np.float32)
    soft = rng.random(slots.size).astype(np.float32)
    vt = np.full((total,), np.nan, np.float32)
    svt = np.full((total,), np.nan, np.float32)
    t_vt, t_svt = torch.from_numpy(vt.copy()), torch.from_numpy(svt.copy())
    ref = v0_core.finalize_trajectory_inplace(t_vt, t_svt, torch.from_numpy(signs), torch.from_numpy(sim),
                                              torch.from_numpy(counts), torch.from_numpy(slots),
                                              torch.from_numpy(res), torch.from_numpy(soft))
    got = oracle.finalize_trajectory_inplace(vt, svt, signs, sim, counts, slots, res, soft)
    for g, r in zip(got, ref):
        assert np.array_equal(g, r.numpy())
    assert np.array_equal(vt, t_vt.numpy(), equal_nan=True)
    assert np.array_equal(svt, t_svt.numpy(), equal_nan=True)


def _fake_net(model_inputs, legal_masks, salt):
    """Deterministic stand-in for the network: priors/values are a hash of the model input."""
    n = model_inputs.shape[0]
    pri = np.zeros((n, 220), np.float32)
    val = np.zeros((n,), np.float32)
    for i in range(n):
        h = hash((model_inputs[i].tobytes(), salt)) & 0xFFFFFFFF
        rng = np.random.default_rng(h)
        p = (rng.random(220).astype(np.float32) + 0.05) * (legal_masks[i] != 0)
        s = p.sum()
        pri[i] = p / s if s > 0 else p
        val[i] = np.float32(rng.random() * 2 - 1)
    return pri, val


@pytest.mark.parametrize("sims,c_puct", [(64, 1.0), (200, 1.5)])
def test_tree_mcts_matches_reference(sims, c_puct):
    """Oracle tree == reference PortableTreeBatch: identical visit counts, Q and root values
    (mirrors tests/v1/test_portable_cpp_mcts.py:203-243), incl. subtree reuse via advance_roots."""
    if REF is None:          # stored: 24 roots x 96 simulations, c_puct 1.25, one move
        return stored.test_tree_mcts_golden()
    _, portable = REF
    st = _collect_playout_states(3, 77, every=9)
    n = st["board"].shape[0]
    ref = portable.PortableTreeBatch([state_obj(st, i) for i in range(n)], exploration_weight=c_puct, num_threads=2)
    mine = oracle.TreeBatch(st, c_puct)
    for move in range(2):
        pr, pm = ref.prepare_roots(), mine.prepare_roots()
        assert np.array_equal(pr["tree_indices"], pm["tree_indices"])
        assert np.array_equal(pr["legal_masks"], pm["legal_masks"])
        assert np.array_equal(pr["model_inputs"], pm["model_inputs"])
        pri, val = _fake_net(pm["model_inputs"], pm["legal_masks"], 0)
        ref.complete_pending(pri, val)
        mine.complete_pending(pri, val)
        for s in range(sims):
            pr, pm = ref.select_leaves(), mine.select_leaves()
            assert np.array_equal(pr["tree_indices"], pm["tree_indices"]), (move, s)
            assert np.array_equal(pr["model_inputs"], pm["model_inputs"]), (move, s)
            assert np.array_equal(pr["legal_masks"], pm["legal_masks"]), (move, s)
            pri, val = _fake_net(pm["model_inputs"], pm["legal_masks"], 1)
            ref.complete_pending(pri, val)
            mine.complete_pending(pri, val)
        ro, mo = ref.root_outputs(), mine.root_outputs()
        assert np.array_equal(ro["visit_counts"], mo["visit_counts"])
        assert np.array_equal(ro["legal_masks"], mo["legal_masks"])
        assert np.array_equal(ro["root_action_values"], mo["root_action_values"])
        assert np.array_equal(ro["root_values"], mo["root_values"])
        assert np.array_equal(ro["terminal"], mo["terminal"])
        assert np.array_equal(ref.root_priors()["priors"], mine.root_priors()["priors"])
        actions = np.where(mo["terminal"] != 0, -1, mo["visit_counts"].argmax(1)).astype(np.int32)
        ref.advance_roots([int(a) for a in actions])
        mine.advance_roots(actions)
