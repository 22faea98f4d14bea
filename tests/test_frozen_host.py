"""FrozenMVSNet refuses, by name, what its kernels cannot run (no GPU needed: the checks come before any device work)."""
import pytest
import torch

import mvs_b200
from mvs_b200 import harness


def test_refuses_a_cpu_module():
    with pytest.raises(mvs_b200.MvsB200Error, match="CPU"):
        mvs_b200.FrozenMVSNet(harness.MVSNet(16, 30.0))


def test_refuses_fp32_precision():
    with pytest.raises(mvs_b200.MvsB200Error, match="fp32"):
        mvs_b200.FrozenMVSNet(harness.MVSNet(16, 30.0, precision="fp32"))


@pytest.mark.parametrize("part", ["feature_encoder", "cost_volume_reg", "depthmap_refine"])
def test_refuses_a_layout_other_than_the_reference(part):
    m = harness.MVSNet(16, 30.0)
    if part == "feature_encoder":
        m.feature_encoder.model[6] = torch.nn.Conv2d(8, 16, 3, stride=2, padding=1, bias=False)     # 3x3 in place of 5x5
    elif part == "cost_volume_reg":
        m.cost_volume_reg.conv_2_1 = torch.nn.Conv3d(32, 32, 3, padding=1, bias=True)
    else:
        del m.depthmap_refine.model[9]                                                           # last convolution gone
    with pytest.raises(mvs_b200.MvsB200Error, match=part.replace("_", ".")):
        mvs_b200.FrozenMVSNet(m)


def test_refuses_a_module_without_the_three_networks():
    with pytest.raises(mvs_b200.MvsB200Error, match="feature_encoder"):
        mvs_b200.FrozenMVSNet(torch.nn.Linear(2, 2))
