"""In-situ CUDA-event timing of the non-convolution kernels of one simulation wave (warm caches, eager launches)."""
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from liuzhou_b200 import native  # noqa: E402
from liuzhou_b200.net import ChessNet, InferenceNet, conv_bf16  # noqa: E402
from liuzhou_b200.tree import encode_inputs  # noqa: E402
from liuzhou_b200.tree_search import TreeMCTS, TreeMCTSConfig  # noqa: E402

n = 4096
dev = torch.device("cuda:0")
torch.manual_seed(20260314)
net = InferenceNet(ChessNet(), dev)
pb = native.PlayoutBatch(n, seed=20260314, device=dev)
pb.run(max_steps=40)
m = TreeMCTS(net, n, TreeMCTSConfig(num_simulations=200, add_dirichlet_noise=False, use_cuda_graph=False), dev)
m.tree.reset(pb.packed, None)
m._root_step()
acc = {}


def timed(name, fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r = fn()
    e1.record()
    acc.setdefault(name, []).append((e0, e1))
    return r


waves = int(sys.argv[1]) if len(sys.argv) > 1 else 160
for w in range(waves):
    tree = m.tree
    timed("select", tree.select_leaves)
    x = m._wave_in
    timed("encode", lambda: encode_inputs(tree.pending_states, "bf16_nhwc", out=x))
    a = timed("trunk (21 convs)", lambda: net.trunk(x))
    t = net.heads._t
    pv = timed("heads conv1x1", lambda: conv_bf16(a, t["conv_wp"], bias=t["conv_bias"], relu1=True)[0])
    timed("heads_tail (+priors)", lambda: net.heads.tail(pv, tree.pending_states, priors_out=m._wave_pri,
                                                          values_out=m._wave_val))
    timed("expand+backup", lambda: tree.complete_pending(m._wave_pri, m._wave_val))
torch.cuda.synchronize()
tot = 0.0
for k, v in acc.items():
    late = [a.elapsed_time(b) * 1e3 for a, b in v[-40:]]
    early = [a.elapsed_time(b) * 1e3 for a, b in v[:20]]
    print(f"{k:24s} first 20 waves {sum(early)/len(early):8.1f} us   last 40 waves {sum(late)/len(late):8.1f} us")
    tot += sum(late) / len(late)
print("sum (last 40):", round(tot, 1), "us")
