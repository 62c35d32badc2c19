"""Which forward path InferenceNet takes for a ChessNet shape and dtype (liuzhou_b200.net.network_path): shape rules
only, so this runs on the CPU with no CUDA device and no native library."""
import pytest
import torch

from liuzhou_b200.net import PATHS, ChessNet, heads_kernel_fits, network_path

BF16 = torch.bfloat16
SMALL = dict(trunk_channels=32, num_blocks=3, policy_channels=16, value_channels=16, value_mlp_channels=32)


@pytest.mark.parametrize("kwargs,dtype,path,heads_fit", [
    ({}, BF16, "trunk", True),                                           # the reference's default network
    ({"num_blocks": 1}, BF16, "trunk", True),
    ({"num_blocks": 11}, BF16, "layered", True),                         # the trunk kernel takes <= 10 blocks
    ({"num_blocks": 12}, BF16, "layered", True),
    ({"num_input_channels": 16}, BF16, "trunk", True),                   # its stem multiplies <= 16 input channels
    ({"num_input_channels": 17}, BF16, "layered", True),
    ({"num_input_channels": 64}, BF16, "layered", True),                 # the per-layer stem pads inputs to 64
    ({"num_input_channels": 65}, BF16, "library", True),
    ({"num_blocks": 0}, BF16, "library", True),
    (SMALL, BF16, "library", True),                                      # 32-wide trunk
    ({"policy_channels": 32}, BF16, "library", True),                    # heads 32 + 64: not one 128-channel conv
    ({"policy_channels": 4, "value_channels": 2}, BF16, "library", False),   # 6 head channels: not a multiple of 8
    ({"value_bucket_bins": 129}, BF16, "library", False),                # heads_tail_kernel takes <= 128 buckets
    ({}, torch.float16, "module", True),                                 # the epilogue kernels are bf16 only
    ({"trunk_channels": 12}, BF16, "module", True),                      # ... in 8-channel vectors
])
def test_default_path_follows_the_shape(kwargs, dtype, path, heads_fit):
    model = ChessNet(**kwargs)
    assert network_path(model, dtype) == path
    assert heads_kernel_fits(model) == heads_fit


def test_explicit_path_must_be_one_the_shape_allows():
    default = ChessNet()
    for p in PATHS:
        assert network_path(default, BF16, p) == p
    deep = ChessNet(num_blocks=12)
    with pytest.raises(ValueError):
        network_path(deep, BF16, "trunk")
    assert network_path(deep, BF16, "layered") == "layered"
    small = ChessNet(**SMALL)
    for p in ("trunk", "layered"):
        with pytest.raises(ValueError):
            network_path(small, BF16, p)
    assert network_path(small, BF16, "library") == "library"
    for p in ("trunk", "layered", "library"):
        with pytest.raises(ValueError):
            network_path(default, torch.float16, p)
    assert network_path(default, torch.float16, "module") == "module"
    with pytest.raises(ValueError):
        network_path(default, BF16, "cudnn")
