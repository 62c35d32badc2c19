"""GPU tests of the search / self-play layer above the kernels: V1RootMCTS.search_batch (root-PUCT mirror),
TreeMCTS (device tree + network) and the self_play_v1_gpu entry with the reference's trajectory format."""
import numpy as np
import pytest
import torch

import oracle
from tests._util import STATE_FIELDS, concat_states, to_torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _np(t):
    return t.detach().cpu().numpy()


def _small_net(seed=7):
    """The reference tests' deterministic tiny network (tests/v1/test_portable_cpp_mcts.py:16-28)."""
    from liuzhou_b200.net import ChessNet

    torch.manual_seed(seed)
    return ChessNet(trunk_channels=8, num_blocks=1, policy_channels=4, value_channels=4, value_mlp_channels=8)


def _playout_states(n_games, seed, every):
    out = []
    for g in range(n_games):
        trace = oracle.random_playout(seed, g, 512, want_trace=True)["trace"]
        st = oracle.initial_states(1)
        for ply, a in enumerate(trace):
            if ply % every == 0:
                out.append(st)
            st = oracle.apply_move_scalar(st, int(a))
    return concat_states(out)


def test_chessnet_matches_reference_architecture():
    from liuzhou_b200.net import ChessNet, flops_per_state

    m = ChessNet()
    n_params = sum(p.numel() for p in m.parameters())
    assert 2_900_000 < n_params < 3_100_000                     # ~3.0 M params (SURVEY 2b)
    assert abs(flops_per_state(m) - 214.5e6) / 214.5e6 < 0.01   # 214.5 MFLOP / state
    keys = set(m.state_dict().keys())
    for k in ("stem_conv.weight", "blocks.9.conv2.weight", "trunk_bn.running_var", "policy_head.gpool_linear.weight",
              "policy_head.out_mark.weight", "value_head.fc2.bias"):
        assert k in keys
    x = torch.zeros(2, 11, 6, 6)
    lp1, lp2, lpm, vl = m.eval()(x)
    assert tuple(lp1.shape) == (2, 36) and tuple(vl.shape) == (2, 101)


def test_root_search_batch_stagewise_vs_oracle():
    """Deterministic configuration (no noise, argmax picks): every stage of search_batch is replayed through the
    oracle from the network outputs recorded on the GPU; visit counts, picks and policy must agree."""
    from liuzhou_b200.mcts_gpu import GpuStateBatch, V1RootMCTS, V1RootMCTSConfig
    from liuzhou_b200.net import InferenceNet, bucket_logits_to_scalar

    st = _playout_states(6, 31, every=5)
    b = st["board"].shape[0]
    net = InferenceNet(_small_net(), DEV, allow_library_convs=True)
    recorded = []
    orig = net.forward

    def rec_forward(x):
        out = orig(x)
        recorded.append([o.clone() for o in out])
        return out

    net.forward = rec_forward
    cfg = V1RootMCTSConfig(num_simulations=64, exploration_weight=1.0, add_dirichlet_noise=False, sample_moves=False)
    mcts = V1RootMCTS(net, cfg, DEV)
    state = GpuStateBatch(*to_torch(st, DEV))
    temps = torch.where(torch.arange(b, device=DEV) % 2 == 0, 1.0, 0.5)
    out = mcts.search_batch(state, temperatures=temps)
    assert len(recorded) == 2
    (lp1, lp2, lpm, rv), (_c1, _c2, _c3, crv) = recorded
    # oracle replay
    mask, meta = oracle.encode_actions_fast(st)
    probs, _ = oracle.project_policy_logits_fast(_np(lp1), _np(lp2), _np(lpm), mask)
    pack = oracle.root_pack_sparse_actions(mask, probs, meta)
    (term, roots, counts, valid_mask, legal_idx, priors, code_mat, flat, codes_all, parents_all) = pack
    children = oracle.batch_apply_moves(st, codes_all, parents_all)
    cvals = _np(bucket_logits_to_scalar(crv).float())
    parent_player = st["current_player"][parents_all]
    leaf = np.where(children["current_player"] == parent_player, cvals, -cvals).astype(np.float32)
    tmask = oracle.terminal_mask_from_next_state(children)
    soft = oracle.soft_value_from_board(children["board"], 2.0)
    leaf = np.where(tmask, soft * np.where(parent_player >= 0, 1.0, -1.0), leaf).astype(np.float32)
    leaf_mat = np.zeros(priors.shape, np.float32)
    leaf_mat.reshape(-1)[flat] = leaf
    visits, value_sum, _ = oracle.root_puct_allocate_visits(priors, leaf_mat, valid_mask, 64, 1.0)
    fin = oracle.root_finalize_from_visits(legal_idx, code_mat, valid_mask, visits, value_sum, roots, b, 220,
                                           _np(temps)[roots])
    assert np.array_equal(_np(out.legal_mask), mask)
    assert np.array_equal(_np(out.terminal_mask), term)
    assert np.array_equal(_np(out.model_input), oracle.states_to_model_input(st))
    # the fp32 projection differs by ~1e-7 between expf implementations; visits are integers and picks follow them
    assert np.array_equal(_np(out.chosen_action_indices), fin[1])
    assert np.array_equal(_np(out.chosen_action_codes), fin[2])
    np.testing.assert_allclose(_np(out.policy_dense), fin[0], rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(_np(out.root_value)[roots], fin[4], rtol=1e-4, atol=1e-5)
    pol = _np(out.policy_dense)
    assert np.allclose(pol[roots].sum(1), 1.0, atol=1e-5) and (pol[~mask] == 0).all()


def test_root_search_noise_and_sampling_invariants():
    from liuzhou_b200.mcts_gpu import GpuStateBatch, V1RootMCTS, V1RootMCTSConfig

    st = _playout_states(6, 32, every=4)
    b = st["board"].shape[0]
    from liuzhou_b200.net import InferenceNet as _IN

    mcts = V1RootMCTS(_IN(_small_net(), DEV, allow_library_convs=True), V1RootMCTSConfig(num_simulations=32), DEV)
    state = GpuStateBatch(*to_torch(st, DEV))
    force = torch.zeros(b, dtype=torch.bool, device=DEV)
    force[::3] = True
    outs = []
    for _ in range(2):
        torch.manual_seed(123)
        outs.append(mcts.search_batch(state, temperatures=1.0, add_dirichlet_noise=True, force_uniform_random_mask=force))
    a, c = outs
    assert torch.equal(a.chosen_action_indices, c.chosen_action_indices) and torch.equal(a.policy_dense, c.policy_dense)
    mask, meta = oracle.encode_actions_fast(st)
    idx = _np(a.chosen_action_indices)
    valid = _np(a.chosen_valid_mask)
    assert (valid == mask.any(1)).all()
    assert all(mask[i, idx[i]] for i in range(b) if valid[i])
    codes = _np(a.chosen_action_codes)
    assert all(np.array_equal(codes[i], meta[i, idx[i]]) for i in range(b) if valid[i])


def test_tree_mcts_search_graph_vs_eager_and_oracle_replay():
    """TreeMCTS with the CUDA-graph wave == eager wave (bit-identical visit counts), and the visit counts equal an
    oracle tree fed with the priors / values the GPU network produced for the same leaves."""
    from liuzhou_b200 import native
    from liuzhou_b200.net import InferenceNet
    from liuzhou_b200.tree_search import TreeMCTS, TreeMCTSConfig

    st = _playout_states(5, 41, every=7)
    n = st["board"].shape[0]
    packed = native.pack_states(to_torch(st, DEV))
    net = InferenceNet(_small_net(), DEV, allow_library_convs=True)
    res = []
    for graph in (True, False):
        cfg = TreeMCTSConfig(num_simulations=48, exploration_weight=1.25, add_dirichlet_noise=False,
                             sample_moves=False, use_cuda_graph=graph)
        out = TreeMCTS(net, n, cfg, DEV).search(packed, temperatures=torch.ones(n, device=DEV))
        res.append(out)
    assert torch.equal(res[0].visit_counts, res[1].visit_counts)
    assert torch.equal(res[0].chosen_action_indices, res[1].chosen_action_indices)
    out = res[0]
    visits = _np(out.visit_counts)
    live = ~_np(out.terminal_mask)
    assert (visits[live].sum(1) == 48).all()
    pol = _np(out.policy_dense)
    assert np.allclose(pol[live].sum(1), 1.0, atol=1e-5)
    np.testing.assert_allclose(pol[live], visits[live] / 48.0, rtol=1e-5, atol=1e-6)   # T = 1 -> N / sum N
    chosen = _np(out.chosen_action_indices)
    assert (visits[live, chosen[live]] == visits[live].max(1)).all()
    # oracle replay with the GPU network as the evaluator: the oracle tree's pending leaf states are evaluated by
    # the same network at the same batch size (row = tree index), so both searches see identical network outputs
    from liuzhou_b200.tree import encode_inputs, heads_to_priors

    def gpu_eval(pend_states, tree_idx):
        full = oracle.initial_states(n)
        for k in STATE_FIELDS:
            full[k][tree_idx] = pend_states[k]
        pk = native.pack_states(to_torch(full, DEV))
        lp1, lp2, lpm, vl = net._forward_eager(encode_inputs(pk, "bf16_nhwc"))
        p, v = heads_to_priors(pk, lp1, lp2, lpm, vl)
        return _np(p)[tree_idx], _np(v)[tree_idx]

    ref = oracle.TreeBatch(st, 1.25)
    pend = ref.prepare_roots()
    ref.complete_pending(*gpu_eval(ref.pending_states(), pend["tree_indices"]))
    for _ in range(48):
        pend = ref.select_leaves()
        ref.complete_pending(*gpu_eval(ref.pending_states(), pend["tree_indices"]))
    ro = ref.root_outputs()
    assert np.array_equal(ro["visit_counts"], visits)
    np.testing.assert_allclose(_np(out.root_value), ro["root_values"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(_np(out.root_action_values), ro["root_action_values"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("backend", ["root", "tree"])
def test_self_play_entry_format_and_determinism(backend):
    """self_play_v1_gpu: reference signature, TensorSelfPlayBatch format (2,692 B / position), finalised value
    targets, policies over legal actions, and bit-identical reruns for a fixed torch seed."""
    from liuzhou_b200.self_play import self_play_v1_gpu

    from liuzhou_b200.net import InferenceNet

    model = InferenceNet(_small_net(), DEV, allow_library_convs=True)
    with pytest.raises(RuntimeError):                   # other network shapes need the explicit library-conv opt-in
        self_play_v1_gpu(_small_net(), num_games=2, mcts_simulations=2, temperature_init=1.0, temperature_final=0.1,
                         temperature_threshold=10, exploration_weight=1.0, device=DEV, search_backend=backend)
    runs = []
    for _ in range(2):
        torch.manual_seed(99)
        batch, stats = self_play_v1_gpu(model, num_games=12, mcts_simulations=8, temperature_init=1.0,
                                        temperature_final=0.1, temperature_threshold=10, exploration_weight=1.0,
                                        device=DEV, add_dirichlet_noise=True, soft_value_k=2.0, max_game_plies=512,
                                        sample_moves=True, concurrent_games=8, search_backend=backend)
        runs.append((batch, stats))
    batch, stats = runs[0]
    n = batch.num_samples
    assert stats.num_games == 12 and stats.num_positions == n and n > 12 * 36
    assert stats.black_wins + stats.white_wins + stats.draws == 12
    assert batch.state_tensors.dtype == torch.float32 and tuple(batch.state_tensors.shape[1:]) == (11, 6, 6)
    assert batch.legal_masks.dtype == torch.bool and tuple(batch.legal_masks.shape) == (n, 220)
    assert batch.policy_targets.dtype == torch.float32 and tuple(batch.policy_targets.shape) == (n, 220)
    assert batch.nbytes() == n * 2692
    vt, svt = _np(batch.value_targets), _np(batch.soft_value_targets)
    assert not np.isnan(vt).any() and not np.isnan(svt).any()
    assert set(np.unique(vt)).issubset({-1.0, 0.0, 1.0}) and (np.abs(svt) <= 1.0).all()
    pol, legal = _np(batch.policy_targets), _np(batch.legal_masks)
    has = legal.any(1)
    assert np.allclose(pol[has].sum(1), 1.0, atol=1e-4) and (pol[~legal] == 0).all()
    planes = _np(batch.state_tensors)
    assert ((planes == 0) | (planes == 1)).all() and (planes[:, 4:11, 0, 0].sum(1) == 1).all()
    assert 36 < stats.avg_game_length <= 512
    assert stats.positions_per_sec > 0 and isinstance(stats.to_dict()["piece_delta_buckets"], dict)
    b2, s2 = runs[1]
    assert torch.equal(batch.policy_targets, b2.policy_targets) and torch.equal(batch.value_targets, b2.value_targets)
    assert torch.equal(batch.state_tensors, b2.state_tensors)


def test_library_path_matches_module_path():
    """The library path -- our fused BatchNorm+ReLU(+residual add) epilogue kernels around the cuDNN convolutions --
    reproduces the plain PyTorch bf16 forward of the module path (bf16 rounding tolerance), with non-trivial
    BatchNorm statistics."""
    from liuzhou_b200.net import ChessNet, InferenceNet

    torch.manual_seed(3)
    model = ChessNet(trunk_channels=32, num_blocks=3, policy_channels=16, value_channels=16, value_mlp_channels=32)
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.normal_(0.0, 0.3)
            m.running_var.uniform_(0.5, 1.5)
            m.weight.data.uniform_(0.5, 1.5)
            m.bias.data.normal_(0.0, 0.2)
    fused = InferenceNet(model, DEV, allow_library_convs=True)
    plain = InferenceNet(model, DEV, path="module", allow_library_convs=True)
    assert fused.trunk is not None and plain.trunk is None
    x = fused.new_input(257)
    x.copy_((torch.rand(257, 11, 6, 6, device=DEV) > 0.6).to(torch.bfloat16))
    a, b = fused._forward_eager(x), plain._forward_eager(x)
    for u, v in zip(a, b):
        torch.testing.assert_close(u, v, rtol=5e-2, atol=5e-2)
    # policy heads are log-probabilities: compare the distributions
    for u, v in zip(a[:3], b[:3]):
        assert float((u.exp() - v.exp()).abs().max()) < 2e-2
    # graph replay == eager
    xin, outs = fused.capture(257, x)
    got = [o.clone() for o in fused.forward(x)]
    for u, v in zip(got, a):
        assert torch.equal(u, v)


@pytest.mark.parametrize("dims", [(32, 16, 16, 32, 101), (128, 64, 64, 128, 101), (8, 4, 4, 8, 101)])
def test_fused_heads_kernel_vs_fp32_pytorch_heads(dims):
    """heads_tail_kernel (fp32 math on the bf16 trunk output) vs the PyTorch head modules evaluated in fp32 on the
    same trunk activations, and forward_priors == heads_to_priors(raw heads)."""
    from liuzhou_b200 import native
    from liuzhou_b200.net import ChessNet, InferenceNet
    from liuzhou_b200.tree import heads_to_priors

    trunk, pc, vc, mlp, bins = dims
    torch.manual_seed(11)
    model = ChessNet(trunk_channels=trunk, num_blocks=1, policy_channels=pc, value_channels=vc,
                     value_mlp_channels=mlp, value_bucket_bins=bins)
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.normal_(0.0, 0.3)
            m.running_var.uniform_(0.5, 1.5)
            m.weight.data.uniform_(0.5, 1.5)
            m.bias.data.normal_(0.0, 0.2)
    net = InferenceNet(model, DEV, allow_library_convs=True)
    if (pc + vc) % 8 != 0:
        assert net.heads is None
        return
    assert net.heads is not None
    st = _playout_states(3, 5, every=2)
    n = st["board"].shape[0]
    if not net.library_convs:                  # the tcgen05 path works on whole 64-board tiles: trim to a multiple of 64
        n = n // 64 * 64
        st = {k: v[:n] for k, v in st.items()}
    packed = native.pack_states(to_torch(st, DEV))
    from liuzhou_b200.tree import encode_inputs

    x = encode_inputs(packed, "bf16_nhwc") if net.library_convs else encode_inputs(packed, "bf16_nhwc",
                                                                                     out=net.new_input(n))
    a = net.trunk(x)
    raw = net.heads(a, want_raw=True)
    if getattr(net, "fused_trunk", False):   # the product path of this network: trunk + heads conv in one kernel
        raw_product = net._forward_eager(x)
        for u, v in zip(raw_product, raw):    # same weights, fp32 instead of bf16 residual stream: close, not equal
            torch.testing.assert_close(u, v, rtol=3e-2, atol=3e-2)
        raw = raw_product
    # fp32 reference heads on the same (bf16) trunk activations
    ref_model = model.to(DEV).float().eval()
    with torch.no_grad():
        af = a.float()
        r1, r2, r3 = ref_model.policy_head(af)
        rv = ref_model.value_head(af)
    # weights were rounded to bf16 for the 1x1 conv and its output is stored in bf16: ~1e-2 abs on log-probs
    for u, v in zip(raw, (r1, r2, r3, rv)):
        torch.testing.assert_close(u, v, rtol=3e-2, atol=3e-2)
    pri, val = net.forward_priors(x, packed)
    pri2, val2 = heads_to_priors(packed, *raw)
    torch.testing.assert_close(pri, pri2, rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(val, val2, rtol=1e-5, atol=1e-6)
    legal = np.zeros((n, 220), bool)
    for i in range(n):
        legal[i, oracle.legal_actions(st, i)[0]] = True
    p = _np(pri)
    assert (p[~legal] == 0).all() and np.allclose(p[legal.any(1)].sum(1), 1.0, atol=1e-5)


def test_tree_search_full_size_properties():
    """BASELINE configs[2] size (4,096 trees x 200 simulations, default 128-channel net on the tcgen05 convs) through
    size-independent properties: every live root receives exactly `sims` visits, visits only on legal actions, the
    policy is a distribution over them, the chosen move is the most visited one, and a second search of the same
    roots reproduces the visit counts bit for bit (no atomics on tree statistics, no noise)."""
    from liuzhou_b200 import native
    from liuzhou_b200.net import ChessNet, InferenceNet
    from liuzhou_b200.tree_search import TreeMCTS, TreeMCTSConfig

    n, sims = 4096, 200
    torch.manual_seed(20260314)
    net = InferenceNet(ChessNet(), DEV)
    chunks = []
    for i, steps in enumerate((0, 9, 30, 45, 70, 100, 140, 200)):
        pb = native.PlayoutBatch(n // 8, seed=99, device=DEV, game_offset=i * (n // 8))
        if steps:
            pb.run(max_steps=steps)
        chunks.append(pb.packed)
    roots = torch.cat(chunks).contiguous()
    mcts = TreeMCTS(net, n, TreeMCTSConfig(num_simulations=sims, add_dirichlet_noise=False, sample_moves=False), DEV)
    temps = torch.ones((n,), device=DEV)
    out1 = mcts.search(roots, temperatures=temps)
    v1 = out1.visit_counts.clone()
    pol1 = out1.policy_dense.clone()
    out2 = mcts.search(roots, temperatures=temps)
    assert torch.equal(v1, out2.visit_counts)
    mcts.tree.check_capacity()
    words, counts = native.legal_masks(roots, scalar_semantics=True)
    legal = native.mask_words_to_bool(words)
    live = ~out1.terminal_mask
    assert int(live.sum()) > n // 2
    assert torch.equal(out1.legal_mask[live], legal[live])
    assert bool((v1[~legal] == 0).all())
    assert bool((v1.sum(1)[live] == sims).all())
    assert torch.allclose(pol1.sum(1)[live], torch.ones_like(pol1.sum(1)[live]), atol=1e-5)
    chosen = out1.chosen_action_indices
    assert bool((chosen[live] >= 0).all()) and bool(legal[live].gather(1, chosen[live].view(-1, 1)).all())
    assert bool((v1[live].gather(1, chosen[live].view(-1, 1)).view(-1) == v1[live].max(1).values).all())
    assert bool((chosen[~live] == -1).all())


def test_tree_mcts_subtree_reuse_across_moves_vs_oracle_replay():
    """TreeMCTS(reuse_subtree=True): search -> advance(chosen) -> search ... over 4 moves (CUDA-graph waves) gives, at
    every move, the visit counts of an oracle tree driven through prepare_roots / select_leaves / advance_roots with
    the same GPU network as evaluator; and the roots the device tree holds are the states the game moved to."""
    from liuzhou_b200 import native
    from liuzhou_b200.net import InferenceNet
    from liuzhou_b200.tree import encode_inputs, heads_to_priors
    from liuzhou_b200.tree_search import TreeMCTS, TreeMCTSConfig

    st = _playout_states(5, 41, every=9)
    n = st["board"].shape[0]
    sims = 40
    net = InferenceNet(_small_net(), DEV, allow_library_convs=True)

    def gpu_eval(pend_states, tree_idx):
        full = oracle.initial_states(n)
        for k in STATE_FIELDS:
            full[k][tree_idx] = pend_states[k]
        pk = native.pack_states(to_torch(full, DEV))
        lp1, lp2, lpm, vl = net._forward_eager(encode_inputs(pk, "bf16_nhwc"))
        p, v = heads_to_priors(pk, lp1, lp2, lpm, vl)
        return _np(p)[tree_idx], _np(v)[tree_idx]

    mcts = TreeMCTS(net, n, TreeMCTSConfig(num_simulations=sims, exploration_weight=1.25, add_dirichlet_noise=False,
                                           sample_moves=False, reuse_subtree=True), DEV)
    ref = oracle.TreeBatch(st, 1.25)
    states = native.pack_states(to_torch(st, DEV))
    inherited = 0
    for move in range(4):
        out = mcts.search(states, temperatures=torch.ones(n, device=DEV))
        pend = ref.prepare_roots()
        if len(pend["tree_indices"]):
            ref.complete_pending(*gpu_eval(ref.pending_states(), pend["tree_indices"]))
        else:
            ref.complete_pending(np.zeros((0, 220), np.float32), np.zeros((0,), np.float32))
        for _ in range(sims):
            pend = ref.select_leaves()
            ref.complete_pending(*gpu_eval(ref.pending_states(), pend["tree_indices"]))
        ro = ref.root_outputs()
        visits = _np(out.visit_counts)
        assert np.array_equal(ro["visit_counts"], visits), move
        live = ~_np(out.terminal_mask)
        if move > 0:
            inherited += int((visits[live].sum(1) > sims).sum())
        chosen = out.chosen_action_indices
        nxt = native.apply_actions(states, chosen.clamp_min(0).to(torch.int32))
        states = torch.where((chosen >= 0).view(-1, 1), nxt, states).contiguous()
        mcts.advance(chosen)
        ref.advance_roots(_np(chosen).astype(np.int32))
        mcts.tree.check_capacity()
        assert torch.equal(mcts.tree.root_states(), states), move
    assert inherited > 0            # some roots really started from inherited visits


def test_stepper_with_subtree_reuse_keeps_roots_in_sync():
    from liuzhou_b200.engine import SelfPlayStepper
    from liuzhou_b200.net import InferenceNet

    net = InferenceNet(_small_net(), DEV, allow_library_convs=True)
    torch.manual_seed(3)
    sp = SelfPlayStepper(net, 256, simulations=24, seed=11, device=DEV, reuse_subtree=True, max_game_plies=40)
    sp.diversify(seed=5, max_random_plies=30, groups=4)
    finished = 0
    for ply in range(14):
        sp.step()
        sp.mcts.tree.check_capacity()
        assert torch.equal(sp.mcts.tree.root_states(), sp.states), ply        # tree roots == game states, restarts incl.
        finished += int(sp._last_done.sum())
        legal, policy = sp.trajectory_block()[1], sp.trajectory_block()[2]
        assert torch.all((policy > 0) <= legal)
    assert finished > 0                                                        # restarts were exercised
    used = sp.mcts.tree.stats()["nodes_used"]
    assert used < 256 * 24 * 40 * 3                                            # compaction bounds the arena


def test_self_play_tree_backend_policy_target_options():
    """policy_target_temperature / policy_target_prior_pseudocount (v1/train.py:2838-2856): with beta > 0 every legal
    action of a stored position carries mass (N + beta * P > 0) and targets are distributions; move selection still
    follows the visit policy (a played move always had visits or was the forced opening pick)."""
    from liuzhou_b200.self_play import self_play_v1_gpu

    torch.manual_seed(5)
    from liuzhou_b200.net import InferenceNet as _IN

    small = _IN(_small_net(), DEV, allow_library_convs=True)
    batch, stats = self_play_v1_gpu(small, num_games=16, mcts_simulations=12, temperature_init=1.0,
                                    temperature_final=0.1, temperature_threshold=6, exploration_weight=1.0, device=DEV,
                                    add_dirichlet_noise=True, max_game_plies=60, sample_moves=True, concurrent_games=16,
                                    search_backend="tree", policy_target_temperature=1.0,
                                    policy_target_prior_pseudocount=2.0)
    pol, legal = batch.policy_targets, batch.legal_masks
    assert stats.num_positions == batch.num_samples > 16 * 20
    assert torch.all((pol > 0) == legal)                               # full legal support, nothing outside
    assert torch.allclose(pol.sum(1), torch.ones(batch.num_samples, device=pol.device), atol=1e-4)
    torch.manual_seed(5)
    base, _ = self_play_v1_gpu(small, num_games=16, mcts_simulations=12, temperature_init=1.0,
                               temperature_final=0.1, temperature_threshold=6, exploration_weight=1.0, device=DEV,
                               add_dirichlet_noise=True, max_game_plies=60, sample_moves=True, concurrent_games=16,
                               search_backend="tree")
    assert not torch.all((base.policy_targets > 0) == base.legal_masks)  # visit-only targets leave unvisited moves at 0


def test_tree_self_play_fast_path_equals_literal_wave_loop():
    """The public tree-backend entry (packed layout, no per-ply host sync, leaf batches compacted to the live games and
    padded to 64-row tiles, value targets broadcast at the end) against the literal reference-style wave loop over the
    drop-in ops (tests/_slow_selfplay.py): identical trajectory batch, bit for bit.  70 games = not a multiple of 64 (the
    padded tile path), default 128-channel network = every convolution on the tcgen05 kernel; deterministic moves."""
    from liuzhou_b200 import _lib
    from liuzhou_b200.net import ChessNet, InferenceNet
    from liuzhou_b200.self_play import self_play_v1_gpu
    from tests._slow_selfplay import slow_tree_self_play

    torch.manual_seed(11)
    net = InferenceNet(ChessNet(), DEV)
    assert not net.library_convs
    ref, ref_len, ref_out = slow_tree_self_play(net, 70, 12, device=DEV)
    batch, stats = self_play_v1_gpu(net, num_games=70, mcts_simulations=12, temperature_init=1.0, temperature_final=0.1,
                                    temperature_threshold=10, exploration_weight=1.0, device=DEV,
                                    add_dirichlet_noise=False, sample_moves=False, concurrent_games=70,
                                    search_backend="tree")
    assert batch.num_samples == ref.num_samples > 70 * 30
    for f in ("state_tensors", "legal_masks", "policy_targets", "value_targets", "soft_value_targets"):
        assert torch.equal(getattr(batch, f), getattr(ref, f)), f
    assert abs(stats.avg_game_length - float(ref_len.float().mean())) < 1e-6
    assert [stats.black_wins, stats.white_wins, stats.draws] == ref_out.tolist()


def test_tree_search_full_size_vs_oracle_three_plies_with_reuse():
    """BASELINE configs[2] at FULL size against the oracle: 4,096 trees x 200 simulations per move, default network on the
    tcgen05 path, three consecutive moves with subtree reuse (advance_roots).  The oracle's tree (restatement of
    PortableTreeBatch, pinned against the reference binary) is fed, wave by wave, the priors / values the GPU network
    produces for ITS pending leaves -- identical visit counts are required on every one of the 4,096 roots after every
    move, and identical chosen moves."""
    from liuzhou_b200 import native
    from liuzhou_b200.net import ChessNet, InferenceNet
    from liuzhou_b200.tree import encode_inputs
    from liuzhou_b200.tree_search import TreeMCTS, TreeMCTSConfig

    n, sims = 4096, 200
    torch.manual_seed(20260314)
    net = InferenceNet(ChessNet(), DEV)
    chunks = []
    for i, steps in enumerate((0, 9, 30, 45, 70, 100, 140, 200)):
        pb = native.PlayoutBatch(n // 8, seed=99, device=DEV, game_offset=i * (n // 8))
        if steps:
            pb.run(max_steps=steps)
        chunks.append(pb.packed)
    roots = torch.cat(chunks).contiguous()
    st = {k: _np(t) for k, t in zip(STATE_FIELDS, native.unpack_states(roots))}
    mcts = TreeMCTS(net, n, TreeMCTSConfig(num_simulations=sims, add_dirichlet_noise=False, sample_moves=False,
                                           reuse_subtree=True), DEV)
    x = net.new_input(n)
    full = {k: np.array(v, copy=True) for k, v in oracle.initial_states(n).items()}

    def gpu_eval(pend_states, tree_idx):
        for k in STATE_FIELDS:
            full[k][tree_idx] = pend_states[k]
        pk = native.pack_states(to_torch(full, DEV))
        encode_inputs(pk, "bf16_nhwc", out=x)
        p, v = net.forward_priors(x, pk)
        return _np(p)[tree_idx], _np(v)[tree_idx]

    def oracle_move(ref):
        pend = ref.prepare_roots()
        if len(pend["tree_indices"]):
            ref.complete_pending(*gpu_eval(ref.pending_states(), pend["tree_indices"]))
        else:
            ref.complete_pending(np.zeros((0, 220), np.float32), np.zeros((0,), np.float32))
        for _ in range(sims):
            pend = ref.select_leaves()
            if len(pend["tree_indices"]):
                ref.complete_pending(*gpu_eval(ref.pending_states(), pend["tree_indices"]))
            else:
                ref.complete_pending(np.zeros((0, 220), np.float32), np.zeros((0,), np.float32))
        return ref.root_outputs()

    ref = oracle.TreeBatch(st, 1.0)
    cur = roots
    temps = torch.ones((n,), device=DEV)
    for move in range(3):
        out = mcts.search(cur, temperatures=temps)
        ro = oracle_move(ref)
        visits = _np(out.visit_counts)
        assert np.array_equal(ro["visit_counts"], visits), (move, int((ro["visit_counts"] != visits).any(1).sum()))
        live = ~_np(out.terminal_mask)
        assert live.sum() > n // 2
        np.testing.assert_allclose(_np(out.root_value)[live], ro["root_values"][live], rtol=1e-5, atol=1e-6)
        chosen = out.chosen_action_indices
        mcts.advance(chosen)
        ref.advance_roots(_np(chosen).astype(np.int32))
        nxt = native.apply_actions(cur, chosen.clamp_min(0).to(torch.int32))
        cur = torch.where((chosen >= 0).view(-1, 1), nxt, cur).contiguous()
    mcts.tree.check_capacity()
