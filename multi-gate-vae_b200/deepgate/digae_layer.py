"""Struct encoder and decoder modules (reference digae_layer.py:26-33, 232-297).

``MultiGCNEncoder`` / ``DirectMultiGCNEncoder`` keep the reference's constructor arguments,
sub-module names (aggr, update, aggr_r, update_r, ln -> checkpoint keys) and forward signatures;
the computation runs in the fused CUDA step kernels of csrc/struct_tc.cu (forward) and csrc/struct_bwd_tc.cu (backward).
"""
import torch
import torch.nn as nn

from . import ops
from .arch.gcn_conv import AggConv
from .schedule import csr_for


class DirectedInnerProductDecoder(nn.Module):
    """sigma(<s[src], t[dst]>)  (reference digae_layer.py:26-33)."""

    def forward(self, s, t, edge_index, sigmoid=True):
        value = (s[edge_index[0]] * t[edge_index[1]]).sum(dim=1)
        return torch.sigmoid(value) if sigmoid else value

    def forward_all(self, s, t, sigmoid=True):
        adj = s @ t.t()
        return torch.sigmoid(adj) if sigmoid else adj


class MultiGCNEncoder(nn.Module):
    def __init__(self, num_rounds, dim_hidden, dim_feature, enable_reverse, layernorm):
        super().__init__()
        self.num_rounds = num_rounds
        self.enable_reverse = True            # the reference forces it (digae_layer.py:237)
        self.layernorm = layernorm
        self.dim_feature = dim_feature
        self.dim_hidden = dim_hidden
        self.aggr = AggConv(dim_hidden, dim_hidden)
        self.update = nn.GRU(dim_hidden + dim_feature, dim_hidden)
        self.aggr_r = AggConv(dim_hidden, dim_hidden)
        self.update_r = nn.GRU(dim_hidden + dim_feature, dim_hidden)
        if layernorm:
            self.ln = nn.LayerNorm(dim_hidden)

    def forward(self, x, edge_index):
        csr = csr_for(edge_index, x.size(0))
        return ops.struct_encoder(x, csr, self.num_rounds, self.layernorm, [self])[0]


class DirectMultiGCNEncoder(nn.Module):
    def __init__(self, dim_feature=3, dim_hidden=128, s_rounds=1, t_rounds=1, enable_reverse=True, layernorm=False):
        super().__init__()
        self.source_conv = MultiGCNEncoder(s_rounds, dim_hidden, dim_feature, enable_reverse, layernorm)
        self.target_conv = MultiGCNEncoder(t_rounds, dim_hidden, dim_feature, enable_reverse, layernorm)

    def forward(self, s, t, edge_index):
        sc, tc = self.source_conv, self.target_conv
        same_input = (s is t) or (s.shape == t.shape and s.data_ptr() == t.data_ptr())
        if same_input and sc.num_rounds == tc.num_rounds and sc.layernorm == tc.layernorm:
            csr = csr_for(edge_index, s.size(0))          # both encoders in one batched launch per step
            out = ops.struct_encoder(s, csr, sc.num_rounds, sc.layernorm, [sc, tc])
            return out[0], out[1]
        return sc(s, edge_index), tc(t, edge_index)
