"""Profiling helper: eager bf16 ChessNet forwards at the wave batch size (run under ncu for a launch list).
usage: profile_forward.py [batch] [warmup iters] [path: trunk | layered | library | module]"""
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from liuzhou_b200.net import ChessNet, InferenceNet  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 3
path = sys.argv[3] if len(sys.argv) > 3 else "trunk"
torch.manual_seed(20260314)
net = InferenceNet(ChessNet(), "cuda:0", path=path, allow_library_convs=True)
x = net.new_input(n)
x.copy_((torch.rand_like(x.float()) > 0.5).to(x.dtype))
for _ in range(iters):
    net._forward_eager(x)
torch.cuda.synchronize()
_, _ = net.capture(n, x)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
net.forward(x)
e0.record()
for _ in range(20):
    net.forward(x)
e1.record()
e1.synchronize()
ms = e0.elapsed_time(e1) / 20
print(f"graph forward n={n} path={path}: {ms:.3f} ms  ({n * net.flops_per_state / ms / 1e9:.1f} TFLOP/s)")
