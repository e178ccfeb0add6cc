"""Image sizes the UNet / VAE convs cannot tile are rejected with a ValueError before anything is launched (no GPU needed)."""
import types

import pytest
import torch

from dreamllm_b200 import ops
from dreamllm_b200.unet import DenoiseLoop, check_planes

SIDES = list(range(256, 1025, 64))


def test_conv_plane_predicate():
    ok = {(h, w) for h in range(1, 130) for w in (1, 2, 4, 8, 16, 32, 64, 128, 256, 384, 512) if ops.conv3x3_plane_supported(h, w)}
    assert (64, 64) in ok and (8, 8) in ok and (4, 4) in ok and (1, 512) in ok and (3, 8) not in ok and (12, 16) not in ok
    assert not ops.conv3x3_plane_supported(16, 96) and not ops.conv3x3_plane_supported(6, 8) and not ops.conv3x3_plane_supported(8, 192)


@pytest.mark.parametrize("height", SIDES)
def test_denoise_loop_rejects_unsupported_sizes_up_front(height):
    unet = types.SimpleNamespace(cfg=dict(block_out_channels=(64, 128, 256, 256)))
    cond = torch.zeros(1, 8, 128)
    for width in SIDES:
        try:
            check_planes(height // 8, width // 8, 4, "UNet")
        except ValueError:
            with pytest.raises(ValueError, match="not supported"):        # raised before the loop touches the (CPU, unusable) model
                DenoiseLoop(unet, cond, 2, 1.0, "ddim", height=height, width=width)
            continue
        assert height in (256, 512, 1024) and width in (256, 512, 1024)
        check_planes(height, width, 4, "VAE")                              # the VAE planes of every UNet-supported size tile as well
