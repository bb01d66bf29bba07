"""CPU restatement of the reference hot path -- TEST INFRASTRUCTURE ONLY.

See oracle/__init__.py for who may import this.  Every function is a plain
PyTorch (CPU, fp32 or fp64) restatement of the algorithm in the cited
reference file:line of Y-Claw/Multilevel-GNN; parameters are passed explicitly
(a ``dict`` with the reference's state_dict key names) so the same tensors can
be fed to the reference modules, to this oracle and to the CUDA drop-ins.
Gradients come from autograd over these compositions.

Pinning: ``tests/test_oracle_pin.py`` checks these functions against
``tests/golden/*.pt`` (outputs of the reference's own files run behind
``oracle/pyg_stub.py`` by ``oracle/make_golden.py``).  The reference itself
ships no golden vectors (SURVEY.md section 4) -- "parity pinned to reference outputs
generated here", not to reference-authored fixtures.

Third-party arithmetic restated here (sources absent from /root/reference;
pins from requirements.txt:147-151): torch-scatter 2.1.0 ``scatter`` /
``scatter_softmax``; torch-geometric 2.2.0 ``MessagePassing.propagate``,
``remove_self_loops`` / ``add_self_loops``, ``degree``, ``DenseSAGEConv``,
``dense_diff_pool``.
"""
import math

import torch
import torch.nn.functional as F


# ----------------------------------------------------------------------------
# segment primitives (torch-scatter 2.1.0 semantics, SURVEY Appendix A)
# ----------------------------------------------------------------------------
def seg_sum(src, index, n):
    """scatter(src, index, dim=0, dim_size=n, reduce='sum')."""
    out = src.new_zeros((n,) + tuple(src.shape[1:]))
    return out.index_add(0, index, src)


def seg_count(index, n, dtype):
    return torch.zeros(n, dtype=dtype, device=index.device).index_add(
        0, index, torch.ones(index.numel(), dtype=dtype, device=index.device))


def seg_mean(src, index, n):
    """reduce='mean': sum / clamp(count, min=1)."""
    cnt = seg_count(index, n, src.dtype).clamp(min=1)
    return seg_sum(src, index, n) / cnt.view(-1, *([1] * (src.dim() - 1)))


def seg_softmax(src, index, n):
    """scatter_softmax: exp(src - max_per_segment) / sum_per_segment, no epsilon."""
    idx = index.view(-1, *([1] * (src.dim() - 1))).expand_as(src)
    mx = src.new_zeros((n,) + tuple(src.shape[1:])).scatter_reduce(0, idx, src, "amax", include_self=False)
    ex = (src - mx.index_select(0, index)).exp()
    den = seg_sum(ex, index, n)
    return ex / den.index_select(0, index)


# ----------------------------------------------------------------------------
# GENConv family
# ----------------------------------------------------------------------------
def gen_message(x, edge_index, edge_attr=None, eps=1e-7):
    """GENConv.message, models/gcn_lib/sparse/torch_vertex.py:94-101.
    x_j = x[edge_index[0]] (PyG source->target flow); relu(x_j + e) + eps."""
    xj = x.index_select(0, edge_index[0])
    if edge_attr is not None:
        xj = xj + edge_attr
    return F.relu(xj) + eps


def gen_aggregate(msg, index, n, aggr="softmax", t=1.0, learn_t=False, p=1.0, y=None):
    """GenMessagePassing.aggregate, models/gcn_lib/sparse/torch_message.py:44-85.

    softmax / softmax_sg / softmax_sum (:49-63): weights = segment softmax of
    t*msg (a constant w.r.t. autograd unless learn_t, :51-55), out = segment sum
    of msg*weights; softmax_sum multiplies by degree**sigmoid(y).
    power / power_sum (:66-80): clamp msg to [1e-7, 10] (in place in the
    reference), segment mean of msg**p, clamp again, **(1/p).
    add / mean / max (:46-47): PyG base aggregation.
    """
    if aggr in ("add", "sum"):
        return seg_sum(msg, index, n)
    if aggr == "mean":
        return seg_mean(msg, index, n)
    if aggr == "max":
        idx = index.view(-1, 1).expand_as(msg)
        return msg.new_zeros(n, msg.shape[1]).scatter_reduce(0, idx, msg, "amax", include_self=False)
    if aggr in ("softmax", "softmax_sg", "softmax_sum"):
        if learn_t and aggr != "softmax_sg":
            w = seg_softmax(msg * t, index, n)
        else:
            with torch.no_grad():
                w = seg_softmax(msg * t, index, n)
        out = seg_sum(msg * w, index, n)
        if aggr == "softmax_sum":
            deg = seg_count(index, n, msg.dtype).unsqueeze(1)
            out = torch.pow(deg, torch.sigmoid(y)) * out
        return out
    if aggr in ("power", "power_sum"):
        lo, hi = 1e-7, 1e1
        m = msg.clamp(lo, hi)
        out = seg_mean(torch.pow(m, p), index, n).clamp(lo, hi)
        out = torch.pow(out, 1 / p)
        if aggr == "power_sum":
            deg = seg_count(index, n, msg.dtype).unsqueeze(1)
            out = torch.pow(deg, torch.sigmoid(y)) * out
        return out
    raise NotImplementedError(aggr)


def msg_norm(x, msg, scale, p=2):
    """MsgNorm.forward, models/gcn_lib/sparse/torch_message.py:175-179."""
    return F.normalize(msg, p=p, dim=1) * x.norm(p=p, dim=1, keepdim=True) * scale


def mlp_forward(sd, prefix, x, norm="batch", act="relu", last_lin=True, training=True, eps_bn=1e-5):
    """MLP(Seq) of Lin / norm / act blocks, models/gcn_lib/sparse/torch_nn.py:54-75.
    Walks the Sequential indices present in ``sd`` under ``prefix``."""
    idxs = sorted({int(k[len(prefix):].split(".")[0]) for k in sd if k.startswith(prefix)})
    lin_idxs = [i for i in idxs if sd[prefix + "%d.weight" % i].dim() == 2]
    for li, i in enumerate(lin_idxs):
        x = F.linear(x, sd[prefix + "%d.weight" % i], sd.get(prefix + "%d.bias" % i))
        last = li == len(lin_idxs) - 1
        if last and last_lin:
            break
        if norm is not None and str(norm).lower() != "none":
            w, b = sd[prefix + "%d.weight" % (i + 1)], sd[prefix + "%d.bias" % (i + 1)]
            if norm == "layer":
                x = F.layer_norm(x, (x.shape[-1],), w, b)
            elif norm == "batch":
                x = F.batch_norm(x, None, None, w, b, True, 0.1, eps_bn)
            else:
                raise NotImplementedError(norm)
        if act == "relu":
            x = F.relu(x)
        elif act == "leakyrelu":
            x = F.leaky_relu(x, 0.2)
    return x


def genconv_forward(sd, x, edge_index, edge_attr, aggr="softmax", t=1.0, learn_t=False, p=1.0,
                    learn_p=False, msg_norm_on=False, encode_edge=False, norm="batch", eps=1e-7,
                    return_parts=False):
    """GENConv.forward, models/gcn_lib/sparse/torch_vertex.py:72-92.
    ``sd`` uses the reference's keys: feature_encoder.{0,1,3}.*, edge_encoder.*,
    msg_norm.msg_scale, t / p / y when learnable."""
    if encode_edge and edge_attr is not None:
        edge_attr = F.linear(edge_attr, sd["edge_encoder.weight"], sd["edge_encoder.bias"])
    t_eff = sd["t"] if "t" in sd else t
    p_eff = sd["p"] if "p" in sd else p
    m = gen_aggregate(gen_message(x, edge_index, edge_attr, eps), edge_index[1], x.shape[0],
                      aggr=aggr, t=t_eff, learn_t=learn_t and "t" in sd, p=p_eff, y=sd.get("y"))
    agg = m
    if msg_norm_on:
        m = msg_norm(x, m, sd["msg_norm.msg_scale"])
    h = x + m
    out = mlp_forward(sd, "feature_encoder.", h, norm=norm, act="relu", last_lin=True)
    if return_parts:
        return out, agg, h
    return out


def pathway_conv_forward(sd, x, edge_index, edge_attr=None, mask=None, aggr="softmax", t=1.0, learn_t=False, norm="batch"):
    """PathwayConv.forward, models/gcn_lib/sparse/torch_vertex.py:155-178 over PathwayMessagePassing.aggregate
    (torch_message.py:124-145, the same arithmetic as GenMessagePassing.aggregate):
      message (:167-175): msg = msg_encoder(flatten(x_j outer edge_attr)) -- a Linear(2*in_dim, in_dim) on the
      [E, in_dim * F_e] outer product, index c * F_e + f -- (no ReLU, no eps: the ``+ self.eps`` line is commented out);
      forward (:155-165): h = x + aggregate(msg); out = relu(mlp(h)); out * mask when a mask is given.
    ``sd``: mlp.{0,1,3}.*, msg_encoder.*, t / y when learnable.  The power modes cannot be constructed in the reference
    (PathwayMessagePassing.__init__ calls super(GenMessagePassing, self), torch_message.py:111: TypeError)."""
    xj = x.index_select(0, edge_index[0])
    if edge_attr is not None:
        msg = torch.matmul(xj[:, :, None], edge_attr[:, None, :]).flatten(1)
    else:
        msg = xj
    msg = F.linear(msg, sd["msg_encoder.weight"], sd["msg_encoder.bias"])
    t_eff = sd["t"] if "t" in sd else t
    m = gen_aggregate(msg, edge_index[1], x.shape[0], aggr=aggr, t=t_eff, learn_t=learn_t and "t" in sd, y=sd.get("y"))
    out = F.relu(mlp_forward(sd, "mlp.", x + m, norm=norm, act="relu", last_lin=True))
    return out * mask if mask is not None else out


# ----------------------------------------------------------------------------
# SAGE / RSAGE (the conv all three shipped configs use)
# ----------------------------------------------------------------------------
def rewrite_self_loops(edge_index, edge_attr, n):
    """remove_self_loops + add_self_loops(fill 1.0), torch_vertex.py:272-273."""
    keep = edge_index[0] != edge_index[1]
    ei = edge_index[:, keep]
    loop = torch.arange(n, dtype=ei.dtype, device=ei.device)
    ei = torch.cat([ei, torch.stack([loop, loop])], dim=1)
    ea = None
    if edge_attr is not None:
        ea = torch.cat([edge_attr[keep], edge_attr.new_ones((n,) + tuple(edge_attr.shape[1:]))], dim=0)
    return ei, ea


def sage_forward(sd, x, edge_index, edge_attr=None, relative=False, act="leakyrelu", normalize=False,
                 prefix="gconv."):
    """SAGEConv.forward/message/update + RSAGEConv, torch_vertex.py:269-304.
    Follows the reference's order: per-EDGE matmul with lin_r.weight.T (:281-285),
    PyG mean aggregation over targets, then nn(cat(x, agg)) (:288-291).
    Note torch_vertex.py:279 guards edge_attr.dim() so edge_attr must not be None there;
    GraphConv always forwards it (None crashes in the reference as well)."""
    n = x.shape[0]
    ei, ea = rewrite_self_loops(edge_index, edge_attr, n)
    if ea is not None and ea.dim() == 1:
        ea = ea.unsqueeze(-1)
    xj = x.index_select(0, ei[0])
    if ea is not None:
        xj = xj * ea
    w = sd[prefix + "lin_r.weight"]
    if relative:
        m = torch.matmul(xj - x.index_select(0, ei[1]), w.t())
    else:
        m = torch.matmul(xj, w.t())
    agg = seg_mean(m, ei[1], n)
    out = mlp_forward(sd, prefix + "nn.", torch.cat((x, agg), dim=1), norm=None, act=act, last_lin=False)
    if normalize:
        out = F.normalize(out, p=2, dim=-1)
    return out


# ----------------------------------------------------------------------------
# MultilevelGNN
# ----------------------------------------------------------------------------
def multilevel_pool(x, gene_pca_match, raw_indice, pca_w, info_mask, nodes_per_graph, n_seg,
                    match_mask=True):
    """Gene -> pathway pool, models/multilevel_gnn.py:212-239.
    x [B*N, C]; gene_pca_match [B, G] (-1 = missing, python negative index wraps in the
    reference: row b*N-1, then zeroed by the mask); raw_indice [B, G] segment ids;
    pca_w [G, P]; info_mask [G, 1].  Returns [B, C, n_seg/3, 3P]."""
    b, g = gene_pca_match.shape
    c = x.shape[1]
    p = pca_w.shape[1]
    idx = gene_pca_match + torch.arange(b, device=x.device)[:, None] * nodes_per_graph
    xg = x[idx]                                                        # [B, G, C]
    if match_mask:
        xg = xg * (gene_pca_match >= 0).to(x.dtype)[:, :, None]
    proj = xg.unsqueeze(3) * (pca_w * info_mask)[None, :, None, :]     # [B, G, C, P]
    proj = proj.permute(0, 2, 1, 3)                                    # [B, C, G, P]
    seg = raw_indice[:, None, :, None].expand(b, c, g, p)
    out = x.new_zeros(b, c, n_seg, p).scatter_add(2, seg, proj)
    return out.reshape(b, c, n_seg // 3, p * 3)


def feature_loss(pca_feature, pca_w, info_mask, pathway_indexs, pca_loss=False, pca_loss_coef=1.0,
                 pca_indep_loss=True):
    """MultilevelGNN.get_feature_loss, models/multilevel_gnn.py:329-348 (including the
    reference's indentation: only the LAST (i, j) pair's |cos| enters indep_loss once per i)."""
    loss = 0
    if pca_loss:
        loss = loss - pca_loss_coef * torch.log(torch.mean(torch.std(pca_feature.reshape(pca_feature.shape[0], -1), dim=0)))
    if pca_indep_loss:
        w = (pca_w * info_mask).detach()
        pdim = w.shape[1]
        ns = int(pathway_indexs.max()) + 1
        indep, count = 0, 0
        for i in range(pdim - 1):
            for j in range(i + 1, pdim):
                count += 1
                mul = seg_sum(w[:, i] * w[:, j], pathway_indexs, ns)
                ln = torch.sqrt(seg_sum(w[:, i] ** 2, pathway_indexs, ns) * seg_sum(w[:, j] ** 2, pathway_indexs, ns))
            indep = indep + torch.mean(torch.abs(mul / (ln + 1e-7)))
        loss = loss + indep / count
    return loss


def multilevel_forward(sd, batch, args, training=False, return_acts=False, pool_arg=None):
    """MultilevelGNN.forward, models/multilevel_gnn.py:132-292, for the configuration family the
    shipped YAMLs select (node_embedding, sage/rsage GraphConv stack, optional dense/res/
    repeat_mask, value_att_mask, linear_projection pool, conv1x1 head).  Dropout layers are
    identity (eval) -- parity runs use eval mode or p=0.
    pool_arg [B, C, Ho, Wo] (optional): the element each max-pool window takes, as the index dh * kw + dw inside the window.
    The pool then gathers that element instead of comparing, so that a window whose two largest values lie within rounding
    of each other takes the same element, and routes its gradient to the same pixel, as the implementation under test."""
    n3 = sd["node_embedding"].shape[0] if "node_embedding" in sd else None
    mask_x = batch.x
    x = batch.x.reshape(-1, 1)
    acts = {}
    if getattr(args, "node_embedding", False):
        x = (x.reshape(-1, n3, 1) * sd["node_embedding"]).reshape(-1, sd["node_embedding"].shape[-1])
    edge_index, edge_attr = batch.edge_index, batch.edge_attr
    if not args.weighted_edge:
        edge_attr = None
    n_layers = len({k.split(".")[1] for k in sd if k.startswith("gnn_model.")})
    feats = []
    for i in range(n_layers):
        y = sage_forward(sd, x, edge_index, edge_attr, relative=(args.gnn_name == "rsage"),
                         act=args.gnn_act, normalize=False, prefix="gnn_model.%d.gconv." % i)
        if args.dense_gnn:
            x = y
            feats.append(x)
        elif args.resgnn:
            x = y + x
        else:
            x = y
        if i + 1 != n_layers and args.repeat_mask and (i + 1) % args.repeat_cyclic == 0:
            if args.repeat_norm:
                x = x / (x ** 2).sum(1).sqrt()[:, None]
            x = x * mask_x.reshape(-1, 1)
        acts["gnn%d" % i] = y          # raw layer output (what a forward hook on gnn_model[i] sees)
    if args.dense_gnn:
        x = torch.cat(feats, dim=-1)
    if args.value_att_mask:
        if args.merge_mode == "mult":
            x = x * mask_x.reshape(-1, 1)
        else:
            x = args.add_coef1 * x + args.add_coef2 * mask_x.reshape(-1, 1)
    pw = sd["learnable_pca_params"]
    x = multilevel_pool(x, batch.gene_pca_match, batch.raw_indice, pw, sd["info_mask"], n3,
                        146 * 3, match_mask=args.pca_match_mask)
    reorder = getattr(batch, "reorder_idxs", None)
    if args.reorder_pathway and reorder is not None:
        x = x[:, :, reorder, :]
    pca_feature = x
    acts["pool"] = x
    conv_keys = sorted({int(k.split(".")[1]) for k in sd if k.startswith("conv_model.")})
    for ci in conv_keys:
        wt = sd["conv_model.%d.weight" % ci]
        x = F.relu(F.conv2d(x, wt, sd["conv_model.%d.bias" % ci], padding=wt.shape[-1] // 2))
    if pool_arg is None:
        x = F.max_pool2d(x, (args.pathway_pool_dim, args.pca_pool_dim))
    else:
        kh, kw = args.pathway_pool_dim, args.pca_pool_dim
        b, c, h, w = x.shape
        ho, wo = h // kh, w // kw
        win = x[:, :, :ho * kh, :wo * kw].reshape(b, c, ho, kh, wo, kw).permute(0, 1, 2, 4, 3, 5).reshape(b, c, ho, wo, kh * kw)
        x = win.gather(4, pool_arg.long().unsqueeze(-1)).squeeze(-1)
    x = torch.flatten(x, start_dim=1)
    if args.use_age:
        x = torch.cat([x, batch.age[:, None]], dim=-1)
    x = F.relu(F.linear(x, sd["head.0.weight"], sd["head.0.bias"]))
    x = F.linear(x, sd["head.3.weight"], sd["head.3.bias"])
    pred = F.softmax(x, dim=1)
    if return_acts:
        return pred, pca_feature, acts
    return pred, pca_feature


def bce_loss(pred, target, weight=None):
    """torch.nn.BCELoss(weight) on softmax outputs, train.py:118,60 (log clamped at -100 like ATen)."""
    l = -(target * torch.log(pred).clamp(min=-100) + (1 - target) * torch.log(1 - pred).clamp(min=-100))
    if weight is not None:
        l = l * weight
    return l.mean()


# ----------------------------------------------------------------------------
# kNN graph construction
# ----------------------------------------------------------------------------
def pairwise_distance(x):
    """models/gcn_lib/sparse/torch_edge.py:53-63 (dense twin dense/torch_edge.py:32-42):
    ||xi||^2 + (-2 xi.xj) + ||xj||^2 with that association."""
    inner = -2 * torch.matmul(x, x.transpose(2, 1))
    sq = torch.sum(x * x, dim=-1, keepdim=True)
    return sq + inner + sq.transpose(2, 1)


def knn_graph_matrix(x, k=16, batch=None):
    """knn_matrix + knn_graph_matrix, sparse/torch_edge.py:66-104.  Row 0 = neighbour ids,
    row 1 = centre ids, both with the per-graph node offset; self is included."""
    bsz = 1 if batch is None else int(batch[-1]) + 1
    xb = x.detach().view(bsz, -1, x.shape[-1])
    _, nn_idx = torch.topk(-pairwise_distance(xb), k=k)
    n = xb.shape[1]
    nn_idx = nn_idx + torch.arange(0, n * bsz, n).view(bsz, 1, 1)
    centre = torch.arange(0, n * bsz).repeat_interleave(k)
    return torch.stack([nn_idx.reshape(-1), centre])


def dense_knn_matrix(x, k=16):
    """dense/torch_edge.py:45-58.  x [B, C, N, 1] -> [2, B, N, k]."""
    xb = x.transpose(2, 1).squeeze(-1).detach()
    b, n, _ = xb.shape
    _, nn_idx = torch.topk(-pairwise_distance(xb), k=k)
    centre = torch.arange(n).view(1, n, 1).expand(b, n, k)
    return torch.stack((nn_idx, centre), dim=0)


def dilate(edge_index, dilation):
    """Dilated.forward deterministic branch, sparse/torch_edge.py:17-29: every d-th column.
    Columns are centre-major with k*d entries per centre, so this keeps ranks 0, d, 2d, ..."""
    return edge_index[:, ::dilation]


def knn_distance_gap(x, k, batch=None):
    """Helper for the kNN parity test: sorted distances to the k+1 nearest, in fp64, so the test
    can tell which neighbour ranks are separated by more than the fp32 evaluation error."""
    bsz = 1 if batch is None else int(batch[-1]) + 1
    xb = x.detach().double().view(bsz, -1, x.shape[-1])
    d = pairwise_distance(xb)
    vals, idx = torch.topk(-d, k=min(k + 1, d.shape[-1]))
    return -vals, idx, d


# ----------------------------------------------------------------------------
# DiffPool
# ----------------------------------------------------------------------------
def dense_sage(sd, prefix, x, adj, normalize=True):
    """PyG 2.2.0 DenseSAGEConv as used at models/diff_pooling.py:24-32,36,45."""
    adj = adj.unsqueeze(0) if adj.dim() == 2 else adj
    out = torch.matmul(adj, x) / adj.sum(dim=-1, keepdim=True).clamp(min=1)
    out = F.linear(out, sd[prefix + "lin_rel.weight"]) + F.linear(x, sd[prefix + "lin_root.weight"], sd[prefix + "lin_root.bias"])
    if normalize:
        out = F.normalize(out, p=2.0, dim=-1)
    return out


def dense_diff_pool(x, adj, s):
    """PyG 2.2.0 dense_diff_pool (called at models/diff_pooling.py:64), mask=None."""
    adj = adj.unsqueeze(0) if adj.dim() == 2 else adj
    s = torch.softmax(s, dim=-1)
    out = torch.matmul(s.transpose(1, 2), x)
    out_adj = torch.matmul(torch.matmul(s.transpose(1, 2), adj), s)
    link = torch.norm(adj - torch.matmul(s, s.transpose(1, 2)), p=2) / adj.numel()
    ent = (-s * torch.log(s + 1e-15)).sum(dim=-1).mean()
    return out, out_adj, link, ent


def diffpool_forward(sd, x, adj, num_layers=2):
    """DiffPool.forward, models/diff_pooling.py:116-133, with after_pooling_layer=1
    (SAGEConvolutions(1, ...) = a single DenseSAGEConv, :28-31,45)."""
    l_tot, e_tot = 0, 0
    for i in range(num_layers):
        s = dense_sage(sd, "diffpool_layers.%d.gnn_pool.layers.0." % i, x, adj)
        z = dense_sage(sd, "diffpool_layers.%d.gnn_embed.layers.0." % i, x, adj)
        x, adj, l, e = dense_diff_pool(z, adj, s)
        x = dense_sage(sd, "after_pool_layers.%d.layers.0." % i, x, adj)
        l_tot = l_tot + l
        e_tot = e_tot + e
    return x, l_tot, e_tot


def predict_head(sd, x, age, args, adj, pca_dim=None):
    """VAE.predict_head, models/vae.py:233-265 (eval mode: dropout = identity).  x [B, C, 146, d];
    ``adj`` = get_pathway_adj() (similarity + I, vae.py:305-306).  Returns (pred, pca_feature, l, e)."""
    l = e = 0
    pca_feature = x
    diff = args.reorder_type == "diff_pooling"

    def sub(prefix):
        return {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}

    if diff and args.diff_pooling_location == "pathway":
        b = x.shape[0]
        x = x.permute(0, 3, 2, 1).reshape(-1, args.pathway_num, args.final_channels)
        x, l, e = diffpool_forward(sub("diff_pooling."), x, adj, num_layers=args.diff_pooling_layer)
        x = x.reshape(b, -1)
    else:
        for ci in sorted({int(k.split(".")[1]) for k in sd if k.startswith("conv_model.")}):
            wt = sd["conv_model.%d.weight" % ci]
            x = F.relu(F.conv2d(x, wt, sd["conv_model.%d.bias" % ci], padding=wt.shape[-1] // 2))
        if diff and args.diff_pooling_location == "head":
            b = x.shape[0]
            x = x.permute(0, 3, 2, 1).reshape(-1, args.pathway_num, args.conv_channel_list[-1])
            x, l, e = diffpool_forward(sub("diff_pooling."), x, adj, num_layers=args.diff_pooling_layer)
            x = x.reshape(b, -1)
        else:
            if args.reorder_type != "no_pooling":
                x = F.max_pool2d(x, (args.pathway_pool_dim, args.pca_pool_dim))
            x = torch.flatten(x, start_dim=1)
    if args.use_age:
        x = torch.cat([x, age[:, None]], dim=-1)
    x = F.relu(F.linear(x, sd["head.0.weight"], sd["head.0.bias"]))
    pred = F.softmax(F.linear(x, sd["head.3.weight"], sd["head.3.bias"]), dim=1)
    return pred, pca_feature, l, e


def foreach_decoder(sd, h):
    """VAE.foreach_decoder, models/vae.py:216-222 with the per-pathway Linear-ReLU-Linear blocks of :54-74."""
    n = len({k.split(".")[1] for k in sd if k.startswith("decoder.")})
    out = []
    for i in range(n):
        z = F.relu(F.linear(h[:, i, :], sd["decoder.%d.0.weight" % i], sd["decoder.%d.0.bias" % i]))
        out.append(F.linear(z, sd["decoder.%d.2.weight" % i], sd["decoder.%d.2.bias" % i]))
    return torch.cat(out, dim=-1)


# ----------------------------------------------------------------------------
# DeeperGCN
# ----------------------------------------------------------------------------
def deepergcn_forward(sd, batch, args, return_hidden=False):
    """DeeperGCN.forward, models/deepergcn.py:185-323, for gnn_encoder='linear', conv='gen',
    no node_embedding, pathway_global_node, pathway_readout='maxpool'; dropout = identity
    (eval / p=0).  Blocks res+ (:232-247), res (:249-258), plain (:263-279)."""
    L, P = args.num_layers, args.pathway_num
    x, ei = batch.x, batch.edge_index
    h = F.linear(x, sd["node_features_encoder.weight"], sd["node_features_encoder.bias"])
    if args.use_edge_attr:
        if args.global_edge == "onehot":
            ee = F.embedding(batch.edge_attr.long(), sd["edge_encoder.weight"])
        else:
            ee = F.linear(batch.edge_attr, sd["edge_encoder.weight"], sd["edge_encoder.bias"])
    else:
        ee = None
    ends = torch.cumsum(batch.node_size, 0).tolist()
    if args.pathway_global_node:
        pe = F.linear(batch.pathway_node_attr, sd["pathway_features_encoder.weight"], sd["pathway_features_encoder.bias"])
        rows = torch.cat([torch.arange(e - P, e) for e in ends])
        h = h.index_copy(0, rows, pe)

    def conv(l, hin):
        sub = {k[len("gcns.%d." % l):]: v for k, v in sd.items() if k.startswith("gcns.%d." % l)}
        return genconv_forward(sub, hin, ei, ee, aggr=args.gcn_aggr, t=args.t, learn_t=args.learn_t,
                               p=args.p, learn_p=args.learn_p, msg_norm_on=args.msg_norm,
                               encode_edge=args.conv_encode_edge, norm=args.norm)

    def nrm(l, hin):
        w, b = sd["norms.%d.weight" % l], sd["norms.%d.bias" % l]
        if args.norm == "layer":
            return F.layer_norm(hin, (hin.shape[-1],), w, b)
        return F.batch_norm(hin, None, None, w, b, True, 0.1, 1e-5)

    if args.block == "res+":
        h = conv(0, h)
        for l in range(1, L):
            h1 = h if args.no_inter_norm else nrm(l - 1, h)
            h = conv(l, F.relu(h1)) + h
        h = nrm(L - 1, h)
    elif args.block == "res":
        h = F.relu(nrm(0, conv(0, h)))
        for l in range(1, L):
            h = F.relu(nrm(l, conv(l, h))) + h
    elif args.block == "plain":
        h = F.relu(nrm(0, conv(0, h)))
        for l in range(1, L):
            h2 = conv(l, h)
            if not args.no_inter_norm:
                h2 = nrm(l, h2)
            h = F.relu(h2) if l != L - 1 else h2
    else:
        raise NotImplementedError(args.block)
    hidden = h
    if args.pathway_global_node:
        pr = torch.stack([h[e - P:e] for e in ends])                  # [B, P, H]
        hg = torch.flatten(F.max_pool1d(pr.transpose(1, 2), 4), start_dim=1)
        if args.pre_concat_age:
            hg = torch.cat([hg, batch.age[:, None]], dim=-1)
        hg = F.relu(F.linear(hg, sd["readout_func.0.weight"], sd["readout_func.0.bias"]))
    else:
        nb = int(batch.batch[-1]) + 1
        hg = seg_mean(h, batch.batch, nb)
    if args.use_age and not args.pre_concat_age:
        hg = torch.cat([hg, batch.age[:, None]], dim=-1)
    keys = sorted({int(k.split(".")[1]) for k in sd if k.startswith("graph_pred_linear.") and k.split(".")[1].isdigit()})
    for j, ki in enumerate(keys):
        hg = F.linear(hg, sd["graph_pred_linear.%d.weight" % ki], sd["graph_pred_linear.%d.bias" % ki])
        if j != len(keys) - 1:
            hg = F.relu(hg)
    out = F.softmax(hg, dim=-1)
    if return_hidden:
        return out, hidden
    return out
