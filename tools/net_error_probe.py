import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from liuzhou_b200.net import ChessNet, InferenceNet  # noqa: E402
DEV = "cuda:0"
for n, blocks in [(64, 1), (192, 2), (4096, 10), (130 * 64, 3)]:
    torch.manual_seed(17)
    model = ChessNet(num_blocks=blocks)
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.normal_(0.0, 0.2); m.running_var.uniform_(0.6, 1.4)
            m.weight.data.uniform_(0.7, 1.3); m.bias.data.normal_(0.0, 0.1)
    net = InferenceNet(model, DEV)
    x = net.new_input(n)
    planes = (torch.rand((n, 11, 6, 6), device=DEV) > 0.6).to(torch.bfloat16)
    x[:, :11] = planes
    fused = [o.clone() for o in net._forward_eager(x)]
    layered = [o.clone() for o in InferenceNet(model, DEV, path="layered")._forward_eager(x)]
    ref = model.to(DEV).float().eval()
    with torch.no_grad():
        out_ref = [o.float() for o in ref(planes.float())]
    ef = max((f.exp() - r.exp()).abs().max().item() for f, r in zip(fused[:3], out_ref[:3]))
    el = max((l.exp() - r.exp()).abs().max().item() for l, r in zip(layered[:3], out_ref[:3]))
    lf = max((f - r).abs().max().item() for f, r in zip(fused[:3], out_ref[:3]))
    vf = (fused[3] - out_ref[3].reshape(fused[3].shape)).abs().max().item()
    vl = (layered[3] - out_ref[3].reshape(fused[3].shape)).abs().max().item()
    vmag = out_ref[3].abs().max().item()
    print(f"n={n} blocks={blocks}: prob err fused {ef:.2e} layered {el:.2e}; log-prob err fused {lf:.2e}; value-logit err fused {vf:.2e} layered {vl:.2e} (|logit| max {vmag:.2f})")
