"""Graph convolution drop-ins (models/gcn_lib/sparse/torch_vertex.py): GENConv :12-104,
SAGEConv/RSAGEConv :226-304, GraphConv :338-363, DynConv and the block wrappers :366-450.
Constructor / forward signatures and state_dict keys are the reference's; the message passing
itself runs in the sm_100a kernels (functional.py)."""
import torch
import torch.nn.functional as F
from torch import nn

from ... import functional as Fn
from ... import graph
from .torch_edge import DilatedKnnGraph
from .torch_message import GenMessagePassing, MsgNorm, PathwayMessagePassing
from .torch_nn import MLP


class GENConv(GenMessagePassing):
    """GENeralized graph convolution: softmax / power-mean aggregation of relu(x_j + e_ji) + eps,
    MsgNorm, residual, then the feature encoder MLP."""

    def __init__(self, in_dim, emb_dim, aggr='softmax', t=1.0, learn_t=False, p=1.0, learn_p=False,
                 y=0.0, learn_y=False, gnn_encoder='linear', msg_norm=False, learn_msg_scale=True,
                 encode_edge=False, bond_encoder=False, edge_feat_dim=None, norm='batch', mlp_layers=2,
                 eps=1e-7, pca_only=False):
        super().__init__(aggr=aggr, t=t, learn_t=learn_t, p=p, learn_p=learn_p, y=y, learn_y=learn_y)
        self.gnn_encoder = gnn_encoder
        if gnn_encoder == 'linear':
            widths = [in_dim] + [in_dim * 2] * (mlp_layers - 1) + [emb_dim]
            self.feature_encoder = MLP(channels=widths, norm=norm, last_lin=True)
        elif gnn_encoder == 'conv1x1':
            self.feature_encoder = nn.Sequential(nn.Conv1d(in_dim, emb_dim, 1), nn.ReLU())
        self.msg_encoder = nn.ReLU()
        self.eps = eps
        self.encode_edge = encode_edge
        self.bond_encoder = bond_encoder
        self.msg_norm = MsgNorm(learn_msg_scale=learn_msg_scale) if msg_norm else None
        if encode_edge:
            if bond_encoder:
                raise NotImplementedError("BondEncoder (OGB molecule leftovers) is out of scope, SURVEY.md section 2 row 4")
            self.edge_encoder = nn.Linear(edge_feat_dim, in_dim)
        self.pca_only = pca_only

    def forward(self, x, edge_index, edge_attr=None):
        if self.pca_only:
            return self.feature_encoder(x)
        if isinstance(edge_attr, Fn.AffineEdge):
            # factored edge term a_e * p + q (DeeperGCN with a scalar edge attribute): this layer's Linear edge encoder is
            # composed analytically and the aggregation kernel rebuilds e_ij in registers -- no [E, H] tensor, no edge GEMM
            ae = edge_attr.compose(self.edge_encoder) if self.encode_edge else edge_attr
            tx = x.flatten(1)
            topo = graph.topology(edge_index, tx.shape[0])
            aggr, t, p, y, learn = self._kernel_args()
            scale = self.msg_norm.msg_scale if self.msg_norm is not None else None
            h = Fn.GenAggregateAffine.apply(tx, ae.a, ae.p, ae.q, t, p, y, scale, topo, aggr, self.eps,
                                            Fn.EPI_MSGNORM if scale is not None else Fn.EPI_RESIDUAL, learn)
            if aggr in ('softmax_sum', 'power_sum'):
                self.sigmoid_y = torch.sigmoid(self.y)
            return self.feature_encoder(h.reshape(x.shape))
        if self.encode_edge and edge_attr is not None:
            edge_emb = Fn.tall_linear(edge_attr, self.edge_encoder)
        else:
            edge_emb = edge_attr
        if edge_emb is None:   # the reference dereferences edge_emb unconditionally (torch_vertex.py:81)
            raise AttributeError("GENConv.forward needs edge_attr (reference: 'NoneType' has no attribute 'flatten')")
        tx, te = x.flatten(1), edge_emb.flatten(1)
        topo = graph.topology(edge_index, tx.shape[0])
        aggr, t, p, y, learn = self._kernel_args()
        if self.msg_norm is not None:
            h = Fn.GenAggregate.apply(tx, te, t, p, y, self.msg_norm.msg_scale, topo, aggr, self.eps,
                                      Fn.EPI_MSGNORM, learn)
        else:
            h = Fn.GenAggregate.apply(tx, te, t, p, y, None, topo, aggr, self.eps, Fn.EPI_RESIDUAL, learn)
        if aggr in ('softmax_sum', 'power_sum'):
            self.sigmoid_y = torch.sigmoid(self.y)
        return self.feature_encoder(h.reshape(x.shape))

    def message(self, x_j, edge_attr=None):
        msg = x_j + edge_attr if edge_attr is not None else x_j
        return self.msg_encoder(msg) + self.eps

    def update(self, aggr_out):
        return aggr_out


class PathwayConv(PathwayMessagePassing):
    """torch_vertex.py:107-178 (the 'multiomix' model's pathway-level convolution): the message of edge j -> i is
    msg_encoder(flatten(x_j outer e_ji)) with msg_encoder = Linear(2 * in_dim, in_dim) (so e has 2 features), aggregated
    by PathwayMessagePassing; out = relu(mlp(x + m)) (* mask).

    The message is linear in x_j for a fixed edge: msg = sum_f e[f] * (W_f x_j) + b with W_f = weight[:, f::F_e].  So the
    node features are transformed ONCE per node (one [N, in] x [in, F_e * in] GEMM instead of a [E, 2 in] x [2 in, in] GEMM
    on the materialised outer products -- E / N times fewer flops and no [E, in * F_e] tensor), the per-edge combination is
    a gather + F_e scaled adds, and the aggregation runs in the segment-softmax kernel on explicit messages
    (GenMessagePassing.aggregate)."""

    def __init__(self, in_dim, emb_dim, aggr='softmax', t=1.0, learn_t=False, p=1.0, learn_p=False, y=0.0, learn_y=False,
                 msg_norm=False, learn_msg_scale=True, encode_edge=False, bond_encoder=False, edge_feat_dim=None,
                 norm='batch', mlp_layers=2, eps=1e-7):
        super().__init__(aggr=aggr, t=t, learn_t=learn_t, p=p, learn_p=learn_p, y=y, learn_y=learn_y)
        self.mlp = MLP(channels=[in_dim] + [in_dim * 2] * (mlp_layers - 1) + [emb_dim], norm=norm, last_lin=True)
        self.msg_encoder = nn.Linear(2 * in_dim, in_dim)
        self.in_dim = in_dim
        self.eps = eps
        self.encode_edge = encode_edge
        self.bond_encoder = bond_encoder
        self.msg_norm = MsgNorm(learn_msg_scale=learn_msg_scale) if msg_norm else None    # built but never applied (:155-165)
        if encode_edge:
            if bond_encoder:
                raise NotImplementedError("BondEncoder (OGB molecule leftovers) is out of scope, SURVEY.md section 2 row 4")
            self.edge_encoder = nn.Linear(edge_feat_dim, in_dim)                          # likewise unused by forward

    def message(self, x_j, edge_attr=None):
        """Reference formulation on gathered rows (kept for callers that use it directly)."""
        msg = torch.matmul(x_j[:, :, None], edge_attr[:, None, :]).flatten(1) if edge_attr is not None else x_j
        return self.msg_encoder(msg)

    def _messages(self, x, edge_index, edge_attr):
        src = edge_index[0]
        if edge_attr is None:
            return self.msg_encoder(x.index_select(0, src))      # shape error for in_dim != 2 * in_dim, as in the reference
        fe = edge_attr.shape[1]
        if fe * self.in_dim != self.msg_encoder.in_features:
            raise RuntimeError("mat1 and mat2 shapes cannot be multiplied (%dx%d and %dx%d)" % (
                edge_attr.shape[0], fe * self.in_dim, self.msg_encoder.in_features, self.in_dim))
        # W[o, c * fe + f] -> Wcat[f * in + o, c]: y[:, f * in + o] = (W_f x)[o]
        wcat = self.msg_encoder.weight.view(self.in_dim, self.in_dim, fe).permute(2, 0, 1).reshape(fe * self.in_dim, self.in_dim)
        if x.is_cuda and x.dim() == 2 and x.shape[0] >= Fn.TallLinear.MIN_ROWS and x.dtype == torch.float32:
            y = Fn.TallLinear.apply(x, wcat.contiguous(), None, False)      # 3xTF32 tensor-core GEMM + mlg_xty weight gradient
        else:
            y = F.linear(x, wcat)
        yj = y.index_select(0, src).view(-1, fe, self.in_dim)
        return (yj * edge_attr.unsqueeze(-1)).sum(1) + self.msg_encoder.bias

    def forward(self, x, edge_index, edge_attr=None, mask=None):
        m = self.aggregate(self._messages(x, edge_index, edge_attr), edge_index[1], dim_size=x.shape[0])
        out = F.relu(self.mlp(x + m))
        return out * mask if mask is not None else out

    def update(self, aggr_out):
        return aggr_out


class SAGEConv(nn.Module):
    """GraphSAGE with edge weights and a rewritten self loop; parameters as in PyG 2.2.0 SAGEConv
    (lin_l is registered but unused by the reference's overridden forward, so it never gets a grad).

    out = nn(cat(x, mean_{j in N(i) U {i}}(w_ij x_j [- x_i]) @ lin_r.weight.T))"""

    def __init__(self, in_channels, out_channels, nn, norm=True, bias=True, relative=False, **kwargs):
        super().__init__()
        if bias:
            raise AttributeError("SAGEConv(bias=True) crashes in the reference too (torch_vertex.py:262-265); "
                                 "RSAGEConv always passes bias=False")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.relative = relative
        self.lin_l = torch.nn.Linear(in_channels, out_channels, bias=False)
        self.lin_r = torch.nn.Linear(in_channels, out_channels, bias=False)
        self.nn = nn
        self.normalize = norm
        self.bias = None

    @property
    def weight(self):
        return self.lin_r.weight.T

    def forward(self, x, edge_index, size=None, edge_attr=None):
        if size is not None:
            raise NotImplementedError("bipartite `size` is never used by the reference models")
        if edge_attr is None:   # torch_vertex.py:279 dereferences edge_attr.dim()
            raise AttributeError("SAGEConv.forward needs edge_attr (reference: 'NoneType' object has no attribute 'dim')")
        if edge_attr.dim() > 1 and edge_attr.shape[-1] != 1:
            raise NotImplementedError("vector edge weights: only [E] / [E,1] edge_attr is used by the reference")
        slope = self._fused_slope()
        # cross-layer activation-backward fusion requested by the model for THIS call (see Fn.SageLayer.forward)
        fuse = getattr(self, "_mlg_fuse", (None, False))
        in_slope, out_premasked = fuse[0], fuse[1]
        link = fuse[2] if len(fuse) > 2 else None      # dict shared with the consumer of this layer's output (next layer / pool)
        prod_link = fuse[3] if len(fuse) > 3 else None # dict shared with the producer of this layer's input
        self._mlg_fuse = (None, False)
        n_total = x.shape[0]
        topo = graph.topology(edge_index, n_total, self_loops=True, edge_weight=edge_attr)
        if isinstance(x, Fn.RankOne):
            # x0 = xs * emb consumed in factored form when the whole layer is fused and the batch is replicated
            if slope is not None and topo.replicas > 1 and topo.n_single == x.emb.shape[0]:
                lin = self.nn[0]
                # with autograd off (MultilevelGNN.predict) no output gradient will ever need masking: the forward kernel then
                # writes no sign bits.  Decided here -- inside a Function's forward the grad mode is always off, and
                # ctx.needs_input_grad follows the inputs' requires_grad, not the caller's grad mode.
                no_backward = not torch.is_grad_enabled()
                return Fn.SageLayer.apply(x.emb, x.xs, self.lin_r.weight, lin.weight, lin.bias, topo, self.relative, slope,
                                          None, out_premasked or no_backward, link, None)
            x = x.materialize()
        x = x.unsqueeze(-1) if x.dim() == 1 else x
        if prod_link is not None and prod_link.get("h1_nm") and slope is None:
            # the producer wrote its rows node-major for a fused consumer, and this call is not fused: back to graph-major
            x = x.view(topo.n_single, -1, x.shape[-1]).transpose(0, 1).reshape(n_total, x.shape[-1])
            prod_link["h1_nm"] = False
        if slope is not None:
            lin = self.nn[0]
            return Fn.SageLayer.apply(x, None, self.lin_r.weight, lin.weight, lin.bias, topo, self.relative, slope,
                                      in_slope, out_premasked, link, prod_link)
        agg_x = Fn.SageAggregate.apply(x, topo, self.relative)
        agg = F.linear(agg_x, self.lin_r.weight)
        return self.update(agg, x)

    def masks_input_grad(self):
        """Whether this layer, asked to, multiplies its input gradient by the producer's activation derivative inside
        its own backward kernel.  Not when it runs transform-first (out_channels < in_channels, Fn.SageLayer): its
        input gradient leaves a GEMM, and the producer applies its own derivative instead."""
        return not self.relative and not (Fn.TRANSFORM_FIRST and self.out_channels < self.in_channels)

    def grad_fusion_slope(self):
        """Slope of this layer's output activation if the layer runs as the fused Fn.SageLayer (so that it can take a
        pre-masked output gradient, and -- when not ``relative`` -- mask its own input gradient); else None."""
        return self._fused_slope()

    def _fused_slope(self):
        """negative slope when ``nn`` is exactly Linear -> ReLU / LeakyReLU (what RSAGEConv builds with
        mlp_norm 'none' and drop 0, i.e. every shipped config) and no output normalisation; else None."""
        if self.normalize or len(self.nn) != 2 or not isinstance(self.nn[0], torch.nn.Linear):
            return None
        act = self.nn[1]
        if isinstance(act, torch.nn.LeakyReLU):
            return float(act.negative_slope)
        if isinstance(act, torch.nn.ReLU):
            return 0.0
        return None

    def update(self, aggr_out, x):
        out = self.nn(torch.cat((x, aggr_out), dim=1))
        if self.normalize:
            out = F.normalize(out, p=2, dim=-1)
        return out


class RSAGEConv(SAGEConv):
    def __init__(self, in_channels, out_channels, act='relu', norm=False, mlp_norm=None, bias=True,
                 relative=False, drop=0.0):
        mlp = MLP([out_channels + in_channels, out_channels], act, mlp_norm, bias, drop=drop)
        super().__init__(in_channels, out_channels, mlp, norm, False, relative)


class GraphConv(nn.Module):
    """Static graph convolution dispatcher; only the conv types a shipped config selects are built
    on kernels ('sage', 'rsage'); the PyG wrappers (edge/mr/gat/gcn/gin) are out of scope (SURVEY section 2 row 2)."""

    def __init__(self, in_channels, out_channels, conv='edge', act='relu', norm=None, bias=True, heads=8,
                 mlp_norm=None, drop=0.0):
        super().__init__()
        kind = conv.lower()
        if kind == 'sage':
            self.gconv = RSAGEConv(in_channels, out_channels, act, norm, mlp_norm, bias, False, drop)
        elif kind == 'rsage':
            self.gconv = RSAGEConv(in_channels, out_channels, act, norm, mlp_norm, bias, True, drop)
        elif kind in ('edge', 'mr', 'gat', 'gcn', 'gin'):
            raise NotImplementedError("conv '%s' wraps torch_geometric layers that no shipped config selects; "
                                      "not part of the hot path" % conv)
        else:
            raise NotImplementedError('conv {} is not implemented'.format(conv))

    def forward(self, x, edge_index, edge_attr=None):
        fuse = self.__dict__.pop("_mlg_fuse", None)     # per-call request from the model, handed to the wrapped conv
        if fuse is not None:
            self.gconv._mlg_fuse = fuse
        return self.gconv(x, edge_index, edge_attr=edge_attr)

    def grad_fusion_slope(self):
        return self.gconv.grad_fusion_slope()

    def masks_input_grad(self):
        return self.gconv.masks_input_grad()

    @property
    def relative(self):
        return self.gconv.relative


class DynConv(GraphConv):
    """Dynamic graph convolution: rebuilds a dilated kNN graph from the features each call."""

    def __init__(self, in_channels, out_channels, kernel_size=9, dilation=1, conv='edge', act='relu',
                 norm=None, bias=True, heads=8, **kwargs):
        super().__init__(in_channels, out_channels, conv, act, norm, bias, heads)
        self.k = kernel_size
        self.d = dilation
        self.dilated_knn_graph = DilatedKnnGraph(kernel_size, dilation, **kwargs)

    def forward(self, x, batch=None, edge_index=None):
        if edge_index is None:
            edge_index = self.dilated_knn_graph(x, batch)
        ones = torch.ones(edge_index.shape[1], 1, device=x.device, dtype=x.dtype)
        return super().forward(x, edge_index, ones)


class PlainDynBlock(nn.Module):
    def __init__(self, channels, kernel_size=9, dilation=1, conv='edge', act='relu', norm=None, bias=True,
                 res_scale=1, **kwargs):
        super().__init__()
        self.body = DynConv(channels, channels, kernel_size, dilation, conv, act, norm, bias, **kwargs)
        self.res_scale = res_scale

    def forward(self, x, batch=None, edge_index=None):
        return self.body(x, batch, edge_index), batch


class ResDynBlock(PlainDynBlock):
    def forward(self, x, batch=None, edge_index=None):
        return self.body(x, batch, edge_index) + x * self.res_scale, batch


class DenseDynBlock(nn.Module):
    def __init__(self, in_channels, out_channels=64, kernel_size=9, dilation=1, conv='edge', act='relu',
                 norm=None, bias=True, **kwargs):
        super().__init__()
        self.body = DynConv(in_channels, out_channels, kernel_size, dilation, conv, act, norm, bias, **kwargs)

    def forward(self, x, batch=None, edge_index=None):
        return torch.cat((x, self.body(x, batch, edge_index)), 1), batch


class ResGraphBlock(nn.Module):
    def __init__(self, channels, conv='edge', act='relu', norm=None, bias=True, heads=8, res_scale=1):
        super().__init__()
        self.body = GraphConv(channels, channels, conv, act, norm, bias, heads)
        self.res_scale = res_scale

    def forward(self, x, edge_index):
        return self.body(x, edge_index) + x * self.res_scale, edge_index


class DenseGraphBlock(nn.Module):
    def __init__(self, in_channels, out_channels, conv='edge', act='relu', norm=None, bias=True, heads=8):
        super().__init__()
        self.body = GraphConv(in_channels, out_channels, conv, act, norm, bias, heads)

    def forward(self, x, edge_index):
        return torch.cat((x, self.body(x, edge_index)), 1), edge_index
