"""Runs only heads_tail_kernel (with priors) a few times on realistic inputs -- for ncu source-level profiling."""
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from liuzhou_b200 import native  # noqa: E402
from liuzhou_b200.net import ChessNet, InferenceNet, conv_bf16  # noqa: E402
from liuzhou_b200.tree import encode_inputs  # noqa: E402

n = 4096
dev = torch.device("cuda:0")
torch.manual_seed(20260314)
net = InferenceNet(ChessNet(), dev)
pb = native.PlayoutBatch(n, seed=20260314, device=dev)
pb.run(max_steps=60)
x = net.new_input(n)
encode_inputs(pb.packed, "bf16_nhwc", out=x)
a = net.trunk(x)
t = net.heads._t
pv = conv_bf16(a, t["conv_wp"], bias=t["conv_bias"], relu1=True)[0]
pri = torch.empty((n, 220), device=dev)
val = torch.empty((n,), device=dev)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
for _ in range(3):
    net.heads.tail(pv, pb.packed, priors_out=pri, values_out=val)
e0.record()
for _ in range(10):
    net.heads.tail(pv, pb.packed, priors_out=pri, values_out=val)
e1.record()
torch.cuda.synchronize()
print(f"heads_tail (+priors): {e0.elapsed_time(e1) * 100:.1f} us")
