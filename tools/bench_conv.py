"""Times our tcgen05 conv (csrc/lz_conv.cu) against cuDNN's fused conv+bias+ReLU and conv + our bn_relu pass
(CUDA-graph replays, CUDA events).  usage: bench_conv.py [n]"""
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from liuzhou_b200.net import bn_relu, conv_bf16, pack_conv_weight  # noqa: E402


def timeit(fn, reps=50):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g.replay()
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


ns = [int(a) for a in sys.argv[1:]] or [4096]
for n in ns:
    cl = torch.channels_last
    x = torch.randn(n, 128, 6, 6, device="cuda", dtype=torch.bfloat16).contiguous(memory_format=cl)
    w = (torch.randn(128, 128, 3, 3, device="cuda", dtype=torch.bfloat16) * 0.03).contiguous(memory_format=cl)
    wp = pack_conv_weight(w)
    b = torch.randn(128, device="cuda", dtype=torch.bfloat16)
    bf = b.float()
    res = torch.randn_like(x)
    sc, sh = torch.rand(128, device="cuda") + 0.5, torch.randn(128, device="cuda")
    o1 = torch.empty_like(x)
    o2 = torch.empty_like(x)
    flop = n * 36 * 128 * 1152 * 2
    t = timeit(lambda: torch.cudnn_convolution_relu(x, w, b, [1, 1], [1, 1], [1, 1], 1))
    print(f"n={n} cuDNN conv+bias+relu          : {t:7.1f} us  {flop / t / 1e6:6.0f} TFLOP/s")
    t = timeit(lambda: conv_bf16(x, wp, bias=bf, relu1=True, out1=o1))
    print(f"n={n} ours  conv+bias+relu          : {t:7.1f} us  {flop / t / 1e6:6.0f} TFLOP/s")
    t = timeit(lambda: bn_relu(res, F.conv2d(x, w, None, 1, 1), sc, sh, True))
    print(f"n={n} cuDNN conv + bn_relu(add,dual): {t:7.1f} us")
    t = timeit(lambda: conv_bf16(x, wp, residual=res, scale=sc, shift=sh, want_out2=True, out1=o1, out2=o2))
    print(f"n={n} ours  conv+residual+bn+relu x2: {t:7.1f} us  {flop / t / 1e6:6.0f} TFLOP/s")
    # back-to-back block: conv1 -> conv2 (what a residual block costs)
    def block_ours():
        h, _ = conv_bf16(x, wp, bias=bf, relu1=True, out1=o1)
        conv_bf16(h, wp, residual=res, scale=sc, shift=sh, want_out2=True, out1=o2, out2=o1)
    def block_cudnn():
        h = torch.cudnn_convolution_relu(x, w, b, [1, 1], [1, 1], [1, 1], 1)
        bn_relu(res, F.conv2d(h, w, None, 1, 1), sc, sh, True)
    print(f"n={n} residual block: cuDNN path {timeit(block_cudnn):7.1f} us   ours {timeit(block_ours):7.1f} us")
