"""Our tcgen05 implicit-GEMM convolution (csrc/lz_conv.cu) vs an fp64 reference of the same op on the same bf16
inputs.  The kernel multiplies bf16 x bf16 exactly, accumulates the K = cin x taps products in fp32 and rounds each
output to bf16 once, so |out - ref| <= 1 bf16 step at the output + K * 2^-24 * sum |x| |w| (c = 1 on both terms).  The
second output reads the first one back: it must be bf16(relu(fmaf(scale, out1, shift))) within one bf16 step."""
import pytest
import torch
import torch.nn.functional as F

from tests._util import bf16_ulp

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U_FP32 = 2.0 ** -24


def _mk(n, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.randn((n, 128, 6, 6), generator=g).to(DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    w = (torch.randn((128, 128, 3, 3), generator=g) * 0.03).to(DEV).to(torch.bfloat16)
    bias = (torch.randn((128,), generator=g) * 0.5).to(DEV)
    res = torch.randn((n, 128, 6, 6), generator=g).to(DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    scale = (torch.rand((128,), generator=g) + 0.5).to(DEV)
    shift = (torch.randn((128,), generator=g) * 0.3).to(DEV)
    return x, w, bias, res, scale, shift


def _conv_ref64(x, w, chunk=2048):
    """fp64 conv2d (stride 1, 'same' padding) and its magnitude sum |x| |w|, both [n, cout, 6, 6]."""
    k = w.size(-1)
    w2 = w.double().reshape(w.size(0), -1).t()
    refs, mags = [], []
    for s in range(0, x.size(0), chunk):
        cols = F.unfold(x[s:s + chunk].double().contiguous(), kernel_size=k, padding=k // 2).transpose(1, 2)
        refs.append((cols @ w2).transpose(1, 2))
        mags.append((cols.abs() @ w2.abs()).transpose(1, 2))
    shape = (x.size(0), w.size(0), 6, 6)
    return torch.cat(refs).reshape(shape), torch.cat(mags).reshape(shape)


def _assert_conv_bound(out, ref, mag, k, what):
    """out (bf16) vs the fp64 ref: one bf16 step of the larger of the two + K * 2^-24 * magnitude."""
    o = out.double()
    bound = bf16_ulp(torch.maximum(o.abs(), ref.abs())) + k * U_FP32 * mag
    diff = (o - ref).abs()
    assert not (diff > bound).any(), (what, int((diff > bound).sum()), float((diff / bound.clamp_min(1e-300)).max()))


def _assert_bn_relu_of(out2, out1, scale, shift, what):
    """out2 == bf16(relu(fmaf(scale, out1, shift))) within one bf16 step (the fp64 product + sum is exact, so its
    fp32 rounding is the fma's)."""
    y = (out1.double() * scale.double().view(1, -1, 1, 1) + shift.double().view(1, -1, 1, 1)).float()
    exp = torch.relu(y).to(torch.bfloat16).double()
    diff = (out2.double() - exp).abs()
    assert not (diff > bf16_ulp(exp)).any(), (what, float(diff.max()))


@pytest.mark.parametrize("n", [64, 192, 4096, 4736, 16384])
def test_conv3x3_bias_relu(n):
    from liuzhou_b200.net import conv_bf16, pack_conv_weight

    x, w, bias, _, _, _ = _mk(n, 1)
    y, _ = conv_bf16(x, pack_conv_weight(w), bias=bias, relu1=True)
    ref, mag = _conv_ref64(x, w)
    b = bias.double().view(1, -1, 1, 1)
    _assert_conv_bound(y, torch.relu(ref + b), mag + b.abs(), 1152, n)


@pytest.mark.parametrize("n", [64, 192, 4736, 16384])
def test_conv_stem_cin64_dual_output(n):
    """The cin = 64, 9-tap instantiation (the stem on the layered path) with the stem epilogue: out1 = relu(conv + bias)
    (stem_bn folded), out2 = relu(bn1_0(out1)).  n = 4,736 is 790 pair tiles of 6 boards over 74 clusters, the last
    one partial."""
    from liuzhou_b200.net import conv_bf16, pack_conv_weight

    g = torch.Generator(device="cpu").manual_seed(n)
    x = torch.randn((n, 64, 6, 6), generator=g)
    x[:, 40:] = (x[:, 40:] > 0.5).float()                           # part of the planes 0 / 1 like the encoded input
    x = x.to(DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    w = (torch.randn((128, 64, 3, 3), generator=g) * 0.05).to(DEV).to(torch.bfloat16)
    bias = (torch.randn((128,), generator=g) * 0.5).to(DEV)
    scale = (torch.rand((128,), generator=g) + 0.5).to(DEV)
    shift = (torch.randn((128,), generator=g) * 0.3).to(DEV)
    out1, out2 = conv_bf16(x, pack_conv_weight(w), bias=bias, relu1=True, scale=scale, shift=shift, want_out2=True)
    ref, mag = _conv_ref64(x, w)
    b = bias.double().view(1, -1, 1, 1)
    _assert_conv_bound(out1, torch.relu(ref + b), mag + b.abs(), 576, n)
    _assert_bn_relu_of(out2, out1, scale, shift, n)
    only2 = conv_bf16(x, pack_conv_weight(w), bias=bias, relu1=True, scale=scale, shift=shift, want_out1=False,
                      want_out2=True)[1]
    assert torch.equal(only2, out2)


@pytest.mark.parametrize("n", [64, 1024])
def test_conv3x3_residual_dual_output(n):
    from liuzhou_b200.net import conv_bf16, pack_conv_weight

    x, w, _, res, scale, shift = _mk(n, 2)
    s, a = conv_bf16(x, pack_conv_weight(w), residual=res, scale=scale, shift=shift, want_out2=True)
    ref, mag = _conv_ref64(x, w)
    _assert_conv_bound(s, ref + res.double(), mag + res.double().abs(), 1152, n)
    _assert_bn_relu_of(a, s, scale, shift, n)                                         # BN reads the stored sum
    only_a = conv_bf16(x, pack_conv_weight(w), residual=res, scale=scale, shift=shift, want_out1=False, want_out2=True)[1]
    assert torch.equal(only_a, a)


def test_conv1x1():
    from liuzhou_b200.net import conv_bf16, pack_conv_weight

    x, w, bias, _, _, _ = _mk(128, 3)
    w1 = w[:, :, 1:2, 1:2].contiguous()
    y, _ = conv_bf16(x, pack_conv_weight(w1), bias=bias, relu1=True)
    ref, mag = _conv_ref64(x, w1)
    b = bias.double().view(1, -1, 1, 1)
    _assert_conv_bound(y, torch.relu(ref + b), mag + b.abs(), 128, "1x1")


def test_conv_is_deterministic_and_border_exact():
    """Zero padding: an all-ones input with all-ones centre-tap-only weights reproduces the input exactly; with
    all nine taps = 1/128 the output counts the in-board neighbours (4 / 6 / 9)."""
    from liuzhou_b200.net import conv_bf16, pack_conv_weight

    n = 64
    x = torch.ones((n, 128, 6, 6), device=DEV, dtype=torch.bfloat16).contiguous(memory_format=torch.channels_last)
    w = torch.full((128, 128, 3, 3), 1.0 / 128.0, device=DEV, dtype=torch.bfloat16)
    y, _ = conv_bf16(x, pack_conv_weight(w))
    cnt = F.conv2d(torch.ones((1, 1, 6, 6), device=DEV), torch.ones((1, 1, 3, 3), device=DEV), None, 1, 1)
    assert torch.equal(y.float(), cnt.expand(n, 128, 6, 6))
    y2, _ = conv_bf16(x, pack_conv_weight(w))
    assert torch.equal(y, y2)


def test_trunk_path_matches_library_path():
    """The whole default ChessNet forward through our tcgen05 convs (20 trunk convs + the heads' 1x1 conv) vs the
    same model built with path="library" (cuDNN conv + bn_relu) on the same inputs: same folded weights, bf16
    activations -> agreement to bf16 noise, and both agree with the fp32 PyTorch module."""
    from liuzhou_b200.net import ChessNet, InferenceNet

    torch.manual_seed(5)
    model = ChessNet()
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.normal_(0.0, 0.2)
            m.running_var.uniform_(0.6, 1.4)
            m.weight.data.uniform_(0.7, 1.3)
            m.bias.data.normal_(0.0, 0.1)
    net = InferenceNet(model, DEV)
    assert net.path == "trunk"
    x64 = net.new_input(128)
    assert x64.size(1) == 64                      # channel-padded input: the stem runs on our conv too
    x = (torch.rand((128, 11, 6, 6), device=DEV) > 0.6).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    x64[:, :11] = x
    out_tc = [o.clone() for o in net._forward_eager(x64)]
    with pytest.raises(RuntimeError):                          # no silent library path: unpadded inputs are refused
        net._forward_eager(x)
    with pytest.raises(RuntimeError):
        net.new_input(100)
    out_pub = net.forward(x.float())                           # the public entry pads rows and channels itself
    for a, b in zip(out_tc, out_pub):
        assert torch.equal(a, b)
    cudnn = InferenceNet(model, DEV, path="library", allow_library_convs=True)
    out_cudnn = [o.clone() for o in cudnn._forward_eager(x)]
    ref = model.to(DEV).float().eval()
    with torch.no_grad():
        out_ref = ref(x.float())
    # measured (tools/net_error_probe.py, 10 blocks, perturbed BatchNorm): log-probs within 3.4e-3 of fp32, value logits
    # within 1.5e-3; the bounds below leave a factor ~6
    for a, b, r in zip(out_tc, out_cudnn, out_ref):
        torch.testing.assert_close(a, b, rtol=0.0, atol=2.5e-2)
        torch.testing.assert_close(a, r.float().reshape(a.shape), rtol=0.0, atol=2e-2)


def test_encode_inputs_channel_padded_layout():
    from liuzhou_b200 import native
    from liuzhou_b200.tree import encode_inputs

    pb = native.PlayoutBatch(256, seed=3, device=DEV)
    pb.run(max_steps=40)
    x11 = encode_inputs(pb.packed, "bf16_nhwc")
    x64 = torch.full((256, 64, 6, 6), 7.0, dtype=torch.bfloat16, device=DEV).contiguous(memory_format=torch.channels_last)
    encode_inputs(pb.packed, "bf16_nhwc", out=x64)
    assert torch.equal(x64[:, :11], x11) and not x64[:, 11:].any()


def _kernel_names(fn):
    """Names of every CUDA kernel launched by fn() (torch.profiler / CUPTI)."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


_LIBRARY_CONV = ("cudnn", "convolve", "nvjet", "cutlass", "xmma", "gemm", "implicit_convolve", "winograd")


def test_no_library_convolution_for_any_batch_size():
    """One convolution path: batches that are not multiples of 64 (a `_split_games` share of 65,311 positions through
    the drop-in `InferenceNet.forward`, a 4,000-game tree search) run on `trunk_kernel` with padded tiles -- not a
    single cuDNN / cuBLAS / CUTLASS kernel is launched (kernel names from torch.profiler)."""
    from liuzhou_b200 import native
    from liuzhou_b200.net import ChessNet, InferenceNet
    from liuzhou_b200.tree_search import TreeMCTS, TreeMCTSConfig

    torch.manual_seed(1)
    net = InferenceNet(ChessNet(), DEV)
    x = (torch.rand((65_311, 11, 6, 6), device=DEV) > 0.6).float()
    net.forward(x)                                                         # warm-up (allocations)
    names = _kernel_names(lambda: net.forward(x))
    assert sum("trunk_kernel" in n for n in names) >= 4                    # 4 chunks of <= 16,384 rows, one launch each
    bad = [n for n in names if any(t in n.lower() for t in _LIBRARY_CONV)]
    assert not bad, sorted(set(bad))[:5]

    n_trees = 4000
    pb = native.PlayoutBatch(n_trees, seed=5, device=DEV)
    pb.run(max_steps=30)
    mcts = TreeMCTS(net, n_trees, TreeMCTSConfig(num_simulations=6, add_dirichlet_noise=False, sample_moves=False), DEV)
    temps = torch.ones((n_trees,), device=DEV)
    out = mcts.search(pb.packed, temperatures=temps)                       # captures the graphs
    assert bool((out.visit_counts.sum(1)[~out.terminal_mask] == 6).all())
    names = _kernel_names(lambda: mcts.search(pb.packed, temperatures=temps))
    assert sum("trunk_kernel" in n for n in names) >= 7                    # root step + 6 waves
    bad = [n for n in names if any(t in n.lower() for t in _LIBRARY_CONV)]
    assert not bad, sorted(set(bad))[:5]
    # the same search with only 1,000 live trees compacts its waves to a 1,024-row batch and gives the same counts
    active = torch.zeros((n_trees,), dtype=torch.bool, device=DEV)
    active[::4] = True
    full = mcts.search(pb.packed, active=active, temperatures=temps)
    mcts.set_live(active)
    compact = mcts.search(pb.packed, active=active, temperatures=temps, live_rows=1000)
    assert mcts._bucket == 1024 and 1024 in mcts.bucket_ladder() and mcts.bucket_for(65) == 128
    mcts.set_live(None)
    assert torch.equal(full.visit_counts, compact.visit_counts)
    assert torch.equal(full.chosen_action_indices, compact.chosen_action_indices)
    assert bool((compact.visit_counts[~active] == 0).all())


@pytest.mark.parametrize("n,blocks", [(64, 1), (192, 2), (4096, 10), (130 * 64, 3)])
def test_trunk_path_matches_layered_path_and_fp32(n, blocks):
    """lzb_trunk_bf16 (whole trunk + heads conv in one persistent kernel, activations resident in shared memory / TMEM,
    fp32 residual stream) against the same model built with path="layered" (one tcgen05 conv per layer, bf16 residual
    stream) and the fp32 PyTorch module on the same positions: the fused kernel must be at least as close to fp32 as
    the per-layer path."""
    from liuzhou_b200.net import ChessNet, InferenceNet

    torch.manual_seed(17)
    model = ChessNet(num_blocks=blocks)
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.normal_(0.0, 0.2)
            m.running_var.uniform_(0.6, 1.4)
            m.weight.data.uniform_(0.7, 1.3)
            m.bias.data.normal_(0.0, 0.1)
    net = InferenceNet(model, DEV)
    assert net.fused_trunk
    x = net.new_input(n)
    planes = (torch.rand((n, 11, 6, 6), device=DEV) > 0.6).to(torch.bfloat16)
    x[:, :11] = planes
    fused = [o.clone() for o in net._forward_eager(x)]
    again = [o.clone() for o in net._forward_eager(x)]
    for a, b in zip(fused, again):
        assert torch.equal(a, b)                                  # deterministic
    layered = [o.clone() for o in InferenceNet(model, DEV, path="layered")._forward_eager(x)]
    ref = model.to(DEV).float().eval()
    with torch.no_grad():
        out_ref = [o.float() for o in ref(planes.float())]
    # measured max-abs errors against the fp32 module (tools/net_error_probe.py): head probabilities 4e-5 .. 1e-4 (fused) vs
    # 5e-5 .. 1.3e-4 (per layer), log-probs <= 3.4e-3, value logits <= 1.5e-3 (fused) vs 1.8e-3 (per layer)
    for f, l, r in zip(fused[:3], layered[:3], out_ref[:3]):
        ef, el = (f.exp() - r.exp()).abs().max().item(), (l.exp() - r.exp()).abs().max().item()
        assert ef <= 5e-4 and ef <= 1.2 * el + 2e-5, (ef, el)
        assert (f.exp() - l.exp()).abs().max().item() <= 5e-4
        assert (f - r).abs().max().item() <= 1.5e-2                              # log-probabilities
    torch.testing.assert_close(fused[3], out_ref[3].reshape(fused[3].shape), rtol=0.0, atol=6e-3)


@pytest.mark.gpu
def test_fused_trunk_copy_handoff_soak():
    """The trunk kernel hands operand copies from the epilogue warps to the MMA thread with a CTA-scope release
    (csrc/lz_trunk.cu: strict_sync off).  A lost or early hand-off would change at least one output element: the same input
    through the kernel 300 times per batch size, while another stream keeps the memory system busy, must give bit-identical
    outputs every time (tools/soak_trunk.py runs 6,000 launches)."""
    from liuzhou_b200.net import ChessNet, InferenceNet

    torch.manual_seed(5)
    net = InferenceNet(ChessNet(), DEV)
    side = torch.cuda.Stream()
    junk = torch.empty(32 << 20, dtype=torch.float32, device=DEV)
    for n in (192, 4096):
        x = net.new_input(n)
        x[:, :11] = (torch.rand((n, 11, 6, 6), device=DEV) > 0.6).to(torch.bfloat16)
        ref = net._trunk_heads_conv(x).clone()
        bad = torch.zeros((), dtype=torch.int64, device=DEV)
        for i in range(300):
            if i % 8 == 0:
                with torch.cuda.stream(side):
                    junk.add_(1.0)
            bad += (net._trunk_heads_conv(x) != ref).any().to(torch.int64)
        torch.cuda.synchronize()
        assert int(bad) == 0, f"{int(bad)} of 300 launches differ at batch {n}"
