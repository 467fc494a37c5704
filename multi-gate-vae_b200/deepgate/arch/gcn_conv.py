"""AggConv parameter holder (reference arch/gcn_conv.py:15-45): msg_i = sum_{j->i} (W h_j + b).
The arithmetic runs inside the fused struct-encoder step kernels (csrc/struct_tc.cu, csrc/struct_bwd_tc.cu)."""
import torch.nn as nn


class AggConv(nn.Module):
    def __init__(self, in_channels, ouput_channels=None, wea=False, mlp=None, reverse=False):
        super().__init__()
        if ouput_channels is None:
            ouput_channels = in_channels
        assert in_channels > 0 and ouput_channels > 0, "The dimension for the AggConv should be larger than 0."
        if wea or mlp is not None:
            raise NotImplementedError("mgv_b200: AggConv edge attributes / custom MLP are not used by any live model")
        self.wea = wea
        self.reverse = reverse
        self.msg = nn.Linear(in_channels, ouput_channels)

    def forward(self, x, edge_index, edge_attr=None, **kwargs):
        raise NotImplementedError(
            "mgv_b200: AggConv is fused into MultiGCNEncoder's CUDA step kernel; call the encoder")
