"""CPU oracle for the level-synchronous DAG message-passing path of
959AI994/Multi-Gate-VAE (DG_VAE/deepgate).

TEST INFRASTRUCTURE -- NOT PRODUCT CODE.  Only ``tests/``, ``__graft_entry__.smoke()``
and ``bench.py``'s CPU-baseline / ``--impl reference`` legs may import this module.
The product package (``multi-gate-vae_b200/deepgate``) never does; it fails loudly
when its CUDA library is missing.

What it is: a plain-PyTorch (CPU, fp32 or fp64) restatement of the reference's
algorithm, written as functions over a ``state_dict`` that uses the reference's
own parameter names (SURVEY.md Appendix A.4), so one set of weights drives the
reference, this oracle and the CUDA implementation.  Every function cites the
reference lines it follows (paths relative to /root/reference/DG_VAE/deepgate).

Pinning: the reference has no tests / golden vectors of its own (SURVEY.md section 4),
so the oracle is pinned against OUTPUTS OF THE REFERENCE ITSELF: the unmodified
reference source is executed in the build container under ``oracle/shim`` by
``oracle/make_golden.py`` and its inputs/outputs/gradients are committed under
``tests/golden/``; ``tests/test_oracle_golden.py`` checks this file against them.

Third-party arithmetic restated here (dependency absent from /root/reference,
un-pinned upstream -- no requirements file; API usage implies PyG 2.0-2.3):
  * torch_geometric.nn.MessagePassing.propagate(aggr='add', flow source->target):
    x_i = x[ei[1]], x_j = x[ei[0]], out = index_add over ei[1] into N rows.
  * torch_geometric.utils.softmax: exp(a - max_group(a).detach()) / (sum_group + 1e-16).
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

# gate code -> module suffix, per model file
GATE_MODULES = {
    "aig": {1: "and", 2: "not"},                                  # dg_ae_model_aig.py:67-68
    "mig": {2: "not", 3: "and", 4: "or", 1: "maj"},               # dg_ae_model_mig.py:79-82
    "xmg": {3: "and", 2: "not", 5: "xor", 1: "maj", 4: "or"},     # dg_ae_model_xmg.py:89-93
    "xag": {3: "and", 2: "not", 5: "xor"},                        # dg_ae_model_xag.py:82-84
}
ENCODER_ATTR = {"aig": "struct_encoder", "mig": "mig_struct_encoder",
                "xmg": "xmg_struct_encoder", "xag": "xag_struct_encoder"}
EPS = 1e-15                                                       # dg_ae_model_mig.py:18


# --------------------------------------------------------------------------- schedule
def top_sort(edge_index, graph_size):
    """ASAP level of every node.  utils/dag_utils.py:10-37 (same peel, same result)."""
    ei = np.asarray(edge_index)
    parent, child = ei[0], ei[1]
    ids = np.arange(graph_size)
    level = np.zeros(graph_size, dtype=np.int64)
    pending = np.ones(graph_size, dtype=bool)
    n = 0
    while pending.any():
        blocked = child[pending[parent]]
        ready = pending & ~np.isin(ids, blocked)
        if not ready.any():
            raise ValueError("cycle in circuit graph (the reference would loop forever)")
        level[ready] = n
        pending[ready] = False
        n += 1
    return torch.from_numpy(level).long()


def return_order_info(edge_index, num_nodes):
    """utils/dag_utils.py:80-88."""
    fl = top_sort(edge_index, num_nodes)
    bl = top_sort(torch.stack([edge_index[1], edge_index[0]]), num_nodes)
    idx = torch.arange(num_nodes, dtype=torch.long)
    return fl, idx, bl, idx.clone()


def subgraph(target_idx, edge_index, dim=1, literal=True):
    """Incoming edges of the target nodes, grouped per target in ``target_idx``
    order, ascending edge id inside a target.  utils/dag_utils.py:91-105.
    ``literal=True`` is the reference's algorithm (one O(E) compare + nonzero per
    node); ``literal=False`` gives the identical result through one stable sort."""
    if literal:
        picks = [(edge_index[dim] == n).nonzero().squeeze(-1) for n in target_idx]
        eids = torch.cat(picks, dim=-1) if picks else torch.zeros(0, dtype=torch.long)
        return edge_index[:, eids]
    key = edge_index[dim]
    rank = torch.full((int(max(int(key.max()) if key.numel() else 0,
                               int(target_idx.max()) if target_idx.numel() else 0)) + 1,),
                      -1, dtype=torch.long)
    rank[target_idx] = torch.arange(target_idx.numel())
    r = rank[key]
    eids = torch.nonzero(r >= 0).squeeze(-1)
    order = torch.sort(r[eids], stable=True).indices
    return edge_index[:, eids[order]]


# --------------------------------------------------------------------------- layers
def linear(P, name, x):
    return F.linear(x, P[name + ".weight"], P[name + ".bias"])


def pyg_softmax(a, index, num_nodes):
    """torch_geometric.utils.softmax as called at arch/tfmlp.py:43 (a is [e, 1])."""
    amax = a.new_full((num_nodes,) + tuple(a.shape[1:]), float("-inf"))
    idx = index.view(-1, *([1] * (a.dim() - 1))).expand_as(a)
    amax = amax.scatter_reduce(0, idx, a.detach(), reduce="amax", include_self=True)
    e = (a - amax.index_select(0, index)).exp()
    denom = torch.zeros((num_nodes,) + tuple(a.shape[1:]), dtype=a.dtype).scatter_add(0, idx, e) + 1e-16
    return e / denom.index_select(0, index)


def tfmlp_aggr(P, name, x, ei):
    """TFMlpAggr.forward / message, arch/tfmlp.py:31-46 (literal q/k/v per edge)."""
    n = x.size(0)
    x_i, x_j = x.index_select(0, ei[1]), x.index_select(0, ei[0])
    q = linear(P, name + ".msg_q", x_i)
    k = linear(P, name + ".msg_k", x_j)
    a = linear(P, name + ".attn_lin", torch.cat([q, k], dim=-1))
    alpha = pyg_softmax(a, ei[1], n)
    t = linear(P, name + ".msg_v", x_j) * alpha
    return torch.zeros(n, t.size(1), dtype=t.dtype).index_add(0, ei[1], t)


def gru_cell(P, name, x, h):
    """torch.nn.GRU, one layer, seq_len 1 (gate order r, z, n).  Call sites:
    dg_ae_model_mig.py:95, digae_layer.py:268-274."""
    gi = F.linear(x, P[name + ".weight_ih_l0"], P[name + ".bias_ih_l0"])
    gh = F.linear(h, P[name + ".weight_hh_l0"], P[name + ".bias_hh_l0"])
    i_r, i_z, i_n = gi.chunk(3, dim=-1)
    h_r, h_z, h_n = gh.chunk(3, dim=-1)
    r = torch.sigmoid(i_r + h_r)
    z = torch.sigmoid(i_z + h_z)
    n = torch.tanh(i_n + r * h_n)
    return (1.0 - z) * n + z * h


def agg_conv(P, name, h, ei):
    """AggConv (aggr='add'), arch/gcn_conv.py:30-42: msg_i = sum_{j->i} (W h_j + b)."""
    m = linear(P, name + ".msg", h.index_select(0, ei[0]))
    return torch.zeros(h.size(0), m.size(1), dtype=m.dtype).index_add(0, ei[1], m)


def multi_gcn_encoder(P, name, x6, ei, rounds, layernorm):
    """MultiGCNEncoder.forward, digae_layer.py:257-277 (enable_reverse forced True :237)."""
    dim = P[name + ".aggr.msg.weight"].size(0)
    dt = P[name + ".aggr.msg.weight"].dtype
    state = torch.ones(x6.size(0), dim, dtype=dt)
    rei = torch.stack([ei[1], ei[0]], dim=0)
    x6 = x6.to(dt)

    def ln(v):
        return F.layer_norm(v, (dim,), P[name + ".ln.weight"], P[name + ".ln.bias"], 1e-5) if layernorm else v

    for _ in range(rounds):
        msg = agg_conv(P, name + ".aggr", state, ei)
        state = ln(gru_cell(P, name + ".update", torch.cat([msg, x6], dim=-1), state))
        msg = agg_conv(P, name + ".aggr_r", state, rei)
        state = ln(gru_cell(P, name + ".update_r", torch.cat([msg, x6], dim=-1), state))
    return state


class _RoundGrad(torch.autograd.Function):
    """Identity whose backward rounds the incoming gradient to ``dtype``."""

    @staticmethod
    def forward(ctx, v, dtype):
        ctx.dtype = dtype
        return v.view_as(v)

    @staticmethod
    def backward(ctx, g):
        return g.to(ctx.dtype).to(g.dtype), None


def multi_gcn_encoder_composed(P, name, x6, ei, rounds, layernorm, round=None):
    """``multi_gcn_encoder`` written the way the struct-encoder kernels compute a step: the GRU pre-activations are one
    product of the tile [sum of neighbour states | h | x | deg | 1] with the AggConv linear composed into the GRU input
    weights (Wc = W_ih[:, :64] W_msg, bc = W_ih[:, :64] b_msg, csrc/pack.cu) and the r / z biases merged.  With
    ``round`` (e.g. torch.bfloat16) every tile operand and weight entry is rounded to that type in the forward
    (straight-through) and the four gate pre-activation gradients (r, z, gi_n, gh_n) are rounded to it in the backward,
    as the low-precision kernels do; everything else stays in the parameters' type."""
    dim = P[name + ".aggr.msg.weight"].size(0)
    dt = P[name + ".aggr.msg.weight"].dtype
    state = torch.ones(x6.size(0), dim, dtype=dt)
    x6 = x6.to(dt)
    ones = torch.ones(x6.size(0), 1, dtype=dt)

    def rnd(v):
        return v if round is None else v + (v.to(round).to(dt) - v).detach()

    def rnd_grad(v):
        return v if round is None else _RoundGrad.apply(v, round)

    def ln(v):
        return F.layer_norm(v, (dim,), P[name + ".ln.weight"], P[name + ".ln.bias"], 1e-5) if layernorm else v

    def step(mod, agg_mod, h, e):
        w_msg, b_msg = P[agg_mod + ".msg.weight"], P[agg_mod + ".msg.bias"]
        w_ih, w_hh = P[mod + ".weight_ih_l0"], P[mod + ".weight_hh_l0"]
        b_ih, b_hh = P[mod + ".bias_ih_l0"], P[mod + ".bias_hh_l0"]
        agg = torch.zeros_like(h).index_add(0, e[1], h.index_select(0, e[0]))
        deg = torch.zeros(h.size(0), 1, dtype=dt).index_add(0, e[1], torch.ones(e.size(1), 1, dtype=dt))
        tile = torch.cat([agg, h, x6, deg, ones], 1)
        # weights over the tile columns agg | h | x | deg of gi = W_ih [msg || x] (msg = W_msg agg + deg b_msg) and gh = W_hh h
        g3, nx = 3 * dim, x6.size(1) + 1
        w_gi = torch.cat([w_ih[:, :dim] @ w_msg, torch.zeros(g3, dim, dtype=dt), w_ih[:, dim:], (w_ih[:, :dim] @ b_msg)[:, None]], 1)
        w_gh = torch.cat([torch.zeros(g3, dim, dtype=dt), w_hh, torch.zeros(g3, nx, dtype=dt)], 1)
        # accumulator columns r | z | gi_n | gh_n; the last tile column carries the biases
        w = torch.cat([w_gi[:2 * dim] + w_gh[:2 * dim], w_gi[2 * dim:], w_gh[2 * dim:]], 0)
        b = torch.cat([b_ih[:2 * dim] + b_hh[:2 * dim], b_ih[2 * dim:], b_hh[2 * dim:]])
        pre = rnd(tile) @ rnd(torch.cat([w, b[:, None]], 1)).t()
        r_pre, z_pre, gi_n, gh_n = (rnd_grad(v) for v in pre.split(dim, 1))
        r, z = torch.sigmoid(r_pre), torch.sigmoid(z_pre)
        n = torch.tanh(gi_n + r * gh_n)
        return ln((1.0 - z) * n + z * h)

    rei = torch.stack([ei[1], ei[0]], dim=0)
    for _ in range(rounds):
        state = step(name + ".update", name + ".aggr", state, ei)
        state = step(name + ".update_r", name + ".aggr_r", state, rei)
    return state


def struct_encoder(P, enc, code, ei, s_rounds, t_rounds, layernorm):
    """DirectMultiGCNEncoder.forward (digae_layer.py:294-297) on the feature the
    models really feed it: one_hot(G.x[:,1], 6) where G.x is already one-hot, i.e.
    one_hot(1{code==1}, 6)  (dg_ae_model_mig.py:71; SURVEY.md Appendix B #1)."""
    feat = F.one_hot((code == 1).long(), num_classes=6)
    s = multi_gcn_encoder(P, enc + ".source_conv", feat, ei, s_rounds, layernorm)
    t = multi_gcn_encoder(P, enc + ".target_conv", feat, ei, t_rounds, layernorm)
    return s, t


# --------------------------------------------------------------------------- model
def model_forward(P, kind, code, edge_index, forward_level, num_rounds=1, s_rounds=4,
                  t_rounds=4, layernorm=True, literal_subgraph=True, hs_override=None, vae_eps=None, stash=None):
    """``Model.forward(G) -> (hs, hf)``.  dg_ae_model_mig.py:64-132 and the aig/xmg/xag
    twins (aig :52-100, xmg :69-150, xag :64-124).  ``code`` is the int gate code per
    node (= G.gate.squeeze(1)); ``forward_level`` as produced by top_sort.
    ``vae_eps = (eps_s, eps_t)``: the variational configuration (BASELINE config 4) -- the struct encoder's (s, t) pass
    through DirectedGVAE.sample (digvae_model.py:134-142, parameters fc_{s,t}_{mu,logstd} in ``P``) before hs_linear and
    (s_mu, s_logstd, t_mu, t_logstd) are appended to ``stash`` for the KL of trainer.py:145-148."""
    enc = ENCODER_ATTR[kind]
    dt = P["hs_linear.weight"].dtype
    n = code.numel()
    if hs_override is None:
        s, t = struct_encoder(P, enc, code, edge_index, s_rounds, t_rounds, layernorm)
        if vae_eps is not None:
            s, t, moments = vae_sample(P, s, t, vae_eps[0].to(dt), vae_eps[1].to(dt))
            if stash is not None:
                stash.append(moments)
        hs = linear(P, "hs_linear", torch.cat([s, t], dim=-1))
    else:
        hs = hs_override
    dim = hs.size(1)
    hf = torch.zeros(n, dim, dtype=dt)
    node_state = torch.cat([hs, hf], dim=-1)
    num_levels = int(forward_level.max().item()) + 1 if n else 1
    ids = torch.arange(n)
    for _ in range(num_rounds):
        for level in range(1, num_levels):
            at_level = forward_level == level
            new_rows = []
            for gcode, suffix in GATE_MODULES[kind].items():
                nodes = ids[at_level & (code == gcode)]
                if nodes.numel() == 0:
                    continue
                sub = subgraph(nodes, edge_index, dim=1, literal=literal_subgraph)
                msg = tfmlp_aggr(P, "aggr_%s_func" % suffix, node_state, sub)
                h_new = gru_cell(P, "update_%s_func" % suffix,
                                 msg.index_select(0, nodes), hf.index_select(0, nodes))
                new_rows.append((nodes, h_new))
            # all types of a level read the pre-level node_state (cat is after the types, mig :129)
            if new_rows:
                hf = hf.clone()
                for nodes, h_new in new_rows:
                    hf[nodes] = h_new
            node_state = torch.cat([hs, hf], dim=-1)
    return hs, hf


def mlp_readout(P, name, x, bn_eps=1e-5):
    """arch/mlp.py:14-56 as built by the models (64->32->32->1, BatchNorm1d, ReLU,
    Dropout 0.2) in eval mode: running statistics, dropout off."""
    for lin, bn in (("0", "1"), ("4", "5")):
        x = F.linear(x, P["%s.fc.%s.weight" % (name, lin)], P["%s.fc.%s.bias" % (name, lin)])
        x = F.batch_norm(x, P["%s.fc.%s.running_mean" % (name, bn)], P["%s.fc.%s.running_var" % (name, bn)],
                         P["%s.fc.%s.weight" % (name, bn)], P["%s.fc.%s.bias" % (name, bn)], False, 0.0, bn_eps)
        x = F.relu(x)
    return F.linear(x, P[name + ".fc.8.weight"], P[name + ".fc.8.bias"])


def pred_prob(P, hf):
    """dg_ae_model_mig.py:134-137."""
    return torch.clamp(mlp_readout(P, "readout_prob", hf), min=0.0, max=1.0)


def recon_loss(P, hs, pos_edge_index, neg_edge_index):
    """dg_ae_model_mig.py:169-191 with the negative edges injected (RNG-free)."""
    s, t = linear(P, "hs_decompose", hs).chunk(2, dim=-1)

    def dec(ei):                                                   # digae_layer.py:26-29
        return torch.sigmoid((s[ei[0]] * t[ei[1]]).sum(dim=1))

    pos, neg = dec(pos_edge_index), dec(neg_edge_index)
    loss = -torch.log(pos + EPS).mean() - torch.log(1 - neg + EPS).mean()
    pred_bin = torch.cat([(pos > 0.5), (neg > 0.5)]).int()
    gt_bin = torch.cat([torch.ones_like(pos), torch.zeros_like(neg)]).int()
    return loss, pred_bin, gt_bin


def zero_normalization(x):
    """utils/utils.py:32-36 (unbiased std)."""
    return (x - torch.mean(x)) / torch.std(x)


def func_loss(hf, tt_pair_index, tt_sim):
    """trainer.py:157-163: L1( z(1 - cos(hf_a, hf_b)), z(tt_sim) )."""
    a, b = hf[tt_pair_index[0]], hf[tt_pair_index[1]]
    dis = 1 - torch.cosine_similarity(a, b, eps=1e-8)
    return F.l1_loss(zero_normalization(dis), zero_normalization(tt_sim.to(dis.dtype)))


def prob_loss(P, hf, prob):
    """trainer.py:154-156."""
    return F.l1_loss(pred_prob(P, hf), prob.to(hf.dtype))


def vae_sample(V, s, t, eps_s, eps_t):
    """DirectedGVAE.sample, digvae_model.py:134-142, with the Gaussian noise injected.
    ``V`` holds fc_{s,t}_{mu,logstd}.{weight,bias}.  Returns samples and the stashed
    (s_mu, s_logstd, t_mu, t_logstd)."""
    s_mu, s_ls = linear(V, "fc_s_mu", s), linear(V, "fc_s_logstd", s)
    t_mu, t_ls = linear(V, "fc_t_mu", t), linear(V, "fc_t_logstd", t)
    return s_mu + torch.exp(s_ls) * eps_s, t_mu + torch.exp(t_ls) * eps_t, (s_mu, s_ls, t_mu, t_ls)


def kl_loss(s_mu, s_ls, t_mu, t_ls, num_nodes):
    """trainer.py:145-148: -0.5/N * mean_i sum_d (1 + 2 logstd - mu^2 - exp(logstd)^2), s plus t."""
    def one(mu, ls):
        return -0.5 / num_nodes * (1 + 2 * ls - mu ** 2 - torch.exp(ls) ** 2).sum(1).mean()
    return one(s_mu, s_ls) + one(t_mu, t_ls)


# --------------------------------------------------------------------------- train step
def train_step_losses(P, kind, G, weights=(1.0, 4.0, 4.0), num_rounds=1, s_rounds=4, t_rounds=4,
                      layernorm=True, literal_subgraph=True, vae_eps=None, kl_weight=0.0):
    """Trainer.run_batch (trainer.py:131-174) + the weighted total (trainer.py:229-231),
    with ``train_pos_edge_index`` / ``neg_edge_index`` taken from ``G`` (the N x N edge
    split of preprocessing.py:56-69 is bypassed on both sides, SURVEY.md section 7 #8).
    ``G`` is a dict: code, edge_index, forward_level, prob, tt_pair_index, tt_sim,
    train_pos_edge_index, neg_edge_index."""
    stash = []
    hs, hf = model_forward(P, kind, G["code"], G["edge_index"], G["forward_level"], num_rounds,
                           s_rounds, t_rounds, layernorm, literal_subgraph, vae_eps=vae_eps, stash=stash)
    rec, _, _ = recon_loss(P, hs, G["train_pos_edge_index"], G["neg_edge_index"])
    prb = prob_loss(P, hf, G["prob"])
    fnc = func_loss(hf, G["tt_pair_index"], G["tt_sim"])
    total = weights[0] * rec + weights[1] * prb + weights[2] * fnc
    parts = {"recon": rec, "prob": prb, "func": fnc, "hs": hs, "hf": hf}
    if stash:
        parts["kl"] = kl_loss(*stash[0], num_nodes=G["code"].numel())
        total = total + kl_weight * parts["kl"]
    return total, parts


# --------------------------------------------------------------------------- parameters
def param_shapes(kind, dim=64, dim_feature=6, layernorm=True, variational=False):
    """Names and shapes of the reference Model's state_dict (SURVEY.md Appendix A.4); ``variational`` adds
    DirectedGVAE's fc_{s,t}_{mu,logstd} (digvae_model.py:111-114)."""
    enc = ENCODER_ATTR[kind]
    sh = {}
    if variational:
        for nme in ("fc_s_mu", "fc_s_logstd", "fc_t_mu", "fc_t_logstd"):
            sh[nme + ".weight"], sh[nme + ".bias"] = (dim, dim), (dim,)
    for conv in ("source_conv", "target_conv"):
        p = "%s.%s" % (enc, conv)
        for a in ("aggr", "aggr_r"):
            sh["%s.%s.msg.weight" % (p, a)] = (dim, dim)
            sh["%s.%s.msg.bias" % (p, a)] = (dim,)
        for u in ("update", "update_r"):
            sh["%s.%s.weight_ih_l0" % (p, u)] = (3 * dim, dim + dim_feature)
            sh["%s.%s.weight_hh_l0" % (p, u)] = (3 * dim, dim)
            sh["%s.%s.bias_ih_l0" % (p, u)] = (3 * dim,)
            sh["%s.%s.bias_hh_l0" % (p, u)] = (3 * dim,)
        if layernorm:
            sh[p + ".ln.weight"] = (dim,)
            sh[p + ".ln.bias"] = (dim,)
    sh["hs_linear.weight"] = (dim, 2 * dim)
    sh["hs_linear.bias"] = (dim,)
    sh["hs_decompose.weight"] = (2 * dim, dim)
    sh["hs_decompose.bias"] = (2 * dim,)
    for suffix in sorted(set(GATE_MODULES[kind].values())):
        a = "aggr_%s_func" % suffix
        sh[a + ".attn_lin.weight"] = (1, 2 * dim)
        sh[a + ".attn_lin.bias"] = (1,)
        for m in ("msg_q", "msg_k", "msg_v"):
            sh["%s.%s.weight" % (a, m)] = (dim, 2 * dim)
            sh["%s.%s.bias" % (a, m)] = (dim,)
        u = "update_%s_func" % suffix
        sh[u + ".weight_ih_l0"] = (3 * dim, dim)
        sh[u + ".weight_hh_l0"] = (3 * dim, dim)
        sh[u + ".bias_ih_l0"] = (3 * dim,)
        sh[u + ".bias_hh_l0"] = (3 * dim,)
    r = "readout_prob.fc"
    sh[r + ".0.weight"], sh[r + ".0.bias"] = (32, dim), (32,)
    sh[r + ".4.weight"], sh[r + ".4.bias"] = (32, 32), (32,)
    sh[r + ".8.weight"], sh[r + ".8.bias"] = (1, 32), (1,)
    for bn in ("1", "5"):
        sh["%s.%s.weight" % (r, bn)] = (32,)
        sh["%s.%s.bias" % (r, bn)] = (32,)
        sh["%s.%s.running_mean" % (r, bn)] = (32,)
        sh["%s.%s.running_var" % (r, bn)] = (32,)
    return sh


def synth_state_dict(kind, seed, dim=64, dim_feature=6, layernorm=True, dtype=torch.float32, variational=False):
    """Reproducible weights (numpy PCG64, independent of torch's init order): every
    matrix/bias ~ U(-1/sqrt(dim), 1/sqrt(dim)) like torch's default GRU/Linear scale;
    norm gains 1 + U(-.1,.1); running_var in [0.5, 1.5].  Keys in sorted order."""
    rng = np.random.default_rng(seed)
    out = {}
    bound = 1.0 / math.sqrt(dim)
    shapes = param_shapes(kind, dim, dim_feature, layernorm)
    extra = {k: v for k, v in param_shapes(kind, dim, dim_feature, layernorm, variational).items() if k not in shapes}
    # the variational head's tensors are drawn AFTER the base set, so a seed gives the same base weights either way
    for name, shape in sorted(shapes.items()) + sorted(extra.items()):
        if name.endswith("running_var"):
            v = 0.5 + rng.random(shape)
        elif name.endswith("running_mean"):
            v = 0.1 * (rng.random(shape) - 0.5)
        elif (".ln." in name or ".fc.1." in name or ".fc.5." in name) and name.endswith("weight"):
            v = 1.0 + 0.2 * (rng.random(shape) - 0.5)
        else:
            v = (2.0 * rng.random(shape) - 1.0) * bound
        out[name] = torch.tensor(v, dtype=dtype)
    return out
