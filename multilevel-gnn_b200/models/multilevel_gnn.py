"""MultilevelGNN drop-in (models/multilevel_gnn.py:13-395 of the reference).

Same constructor (``args`` namespace, opt.py flags), same ``forward(input_batch, ...) -> (pred,
pca_feature)``, same setters and state_dict keys (node_embedding, learnable_pca_params, info_mask,
gnn_model.{i}.gconv.*, conv_model.{0,2}.*, head.{0,3}.*).  The level-1 message passing (GraphConv
'sage'/'rsage' stack), the embed-scale prologue and the gene->pathway pool run in the sm_100a
kernels; the 1x1-conv / MLP head stays in torch (SURVEY.md section 8f row 2, "next").
"""
import torch
import torch.nn as nn

from .. import functional as Fn
from .. import graph
from ..gcn_lib.sparse.torch_vertex import GraphConv


class MultilevelGNN(nn.Module):
    GENES = 5135      # reference hard-codes node_num (multilevel_gnn.py:34)
    SLOTS = 25015     # and the gene-slot count (multilevel_gnn.py:74)
    FUSE_ACT_BACKWARD = True     # cross-layer activation-backward fusion (see forward); False = one pass per layer

    def __init__(self, args, pca_params=None, pathway_indexs=None):
        super().__init__()
        self.args = args
        self.pca_compare = args.pca_compare
        self.pca_prelinear = args.pca_prelinear
        self.learnable_pca = args.learnable_pca
        self.pca_loss = args.pca_loss
        self.pca_indep_loss = args.pca_indep_loss
        self.pca_dim = args.pca_dim
        self.pathway_pool_dim = args.pathway_pool_dim
        self.pca_pool_dim = args.pca_pool_dim
        self.pathway_indexs = None
        self.reorder_idxs = None
        self.mutual_info_mask = args.mutual_info_mask
        self.mutual_info_threshold = args.mutual_info_threshold
        self.pca_loss_coef = args.pca_loss_coef
        self.node_select_threshold = args.node_select_threshold
        self.mutual_neighbors = args.mutual_neighbors
        self.node_num = self.GENES
        self.mutual_info_mask_cache = {}
        self.head_dim = args.head_dim
        self.epoch = None
        self.step = None
        self.used_omics = args.used_omics
        if self.pca_compare or self.pca_prelinear:
            raise NotImplementedError("pca_compare / pca_prelinear heads are not selected by any shipped config")
        if args.reduction_method != "linear_projection":
            raise NotImplementedError("reduction_method=%s (torch.svd / pca_lowrank) is out of scope, SURVEY.md section 2 row 16"
                                      % args.reduction_method)
        if len(self.used_omics) != 3:
            raise NotImplementedError("used_omics subsets are not selected by any shipped config")

        self.input_drop = nn.Dropout(p=args.input_drop) if args.input_drop is not None else None
        self.input_emb_drop = nn.Dropout(p=args.input_emb_drop) if args.input_emb_drop is not None else None

        if args.node_embedding:
            self.node_embedding = nn.Parameter(torch.rand([self.node_num * 3, args.node_embedding_dim]),
                                               requires_grad=not args.freeze_node_embedding)
            init = args.embedding_init_type
            if init == "xavier":
                nn.init.xavier_uniform_(self.node_embedding)
            elif init == "ones":
                nn.init.constant_(self.node_embedding, 1)
            elif init == "constant":
                nn.init.constant_(self.node_embedding, args.emb_val)
            elif init == "uniform":
                nn.init.uniform_(self.node_embedding)
            self.node_embedding_dim = args.node_embedding_dim
        else:
            self.node_embedding = None
            self.node_embedding_dim = 1

        conv_kw = dict(act=args.gnn_act, conv=args.gnn_name, mlp_norm=args.gnn_mlp_norm, drop=args.gnn_dropout)
        blocks = [GraphConv(self.node_embedding_dim, args.hidden_channels, **conv_kw)]
        for _ in range(args.num_layers - 2):
            blocks.append(GraphConv(args.hidden_channels, args.hidden_channels, **conv_kw))
        blocks.append(GraphConv(args.hidden_channels, args.final_channels, heads=args.final_head,
                                norm=args.gnn_last_norm, **conv_kw))
        self.gnn_model = nn.ModuleList(blocks)

        self.learnable_pca_params = nn.Parameter(torch.rand([self.SLOTS, self.pca_dim]),
                                                 requires_grad=not args.freeze_pca_weight)
        if pca_params is None:
            if args.pca_init_type is None:
                nn.init.xavier_uniform_(self.learnable_pca_params.data)
            elif args.pca_init_type == "orthogonal":
                nn.init.orthogonal_(self.learnable_pca_params.data)
        else:
            self.learnable_pca_params.data = pca_params

        # NOTE: like the reference, the constructor rewrites args.final_channels in these two modes
        if args.edge_type == 'merge':
            args.final_channels *= 2
        if args.dense_gnn:
            args.final_channels = (args.num_layers - 1) * args.hidden_channels + args.final_channels

        convs, cin = [], args.final_channels
        for cout, ks in zip(args.conv_channel_list, args.conv_kernel_list):
            convs += [nn.Conv2d(cin, cout, ks, padding=ks // 2), nn.ReLU()]
            cin = cout
        self.conv_model = nn.ModuleList(convs)
        self.pooling = nn.MaxPool2d((self.pathway_pool_dim, self.pca_pool_dim))
        self.drop1 = nn.Dropout(0.25 if args.feature_drop else 0)
        head_in = (args.conv_channel_list[-1] * (146 // self.pathway_pool_dim)
                   * ((len(self.used_omics) * self.pca_dim) // self.pca_pool_dim) + (1 if args.use_age else 0))
        self.head = nn.Sequential(nn.Linear(head_in, self.head_dim), nn.ReLU(), nn.Dropout(0.5),
                                  nn.Linear(self.head_dim, 2), nn.Softmax(dim=1))
        self.init_weight()

    # ------------------------------------------------------------------------------------------
    def pool_genes(self, input_batch, x=None, gene_pca_match=None, raw_indice=None, value_mask=True, fused=False):
        """Level 1 -> level 2 (models/multilevel_gnn.py:140-239): embed-scale, the GraphConv stack on the gene graph, the
        value mask and the gene -> pathway projection pool.  Returns the pooled tensor [B, C, 438, P] (a permuted view of the
        channel-last buffer the pool kernel writes).  ``value_mask=False``: the VAE encoder's variant (models/vae.py:128-190,
        where the mask lines are commented out).  ``fused``: take the fused layer chain even when autograd records nothing
        (``predict``); by default it is taken only when it does."""
        args = self.args
        if x is not None:
            mask_x = x
        else:
            mask_x = input_batch.x
            gene_pca_match = input_batch.gene_pca_match
            raw_indice = input_batch.raw_indice
        x = mask_x.reshape(-1, 1)
        if self.input_drop is not None:
            x = self.input_drop(x)
        n3 = self.node_num * 3
        xs = x                                                       # [B*N, 1] scalar node values

        edge_index, edge_attr = input_batch.edge_index, input_batch.edge_attr
        if isinstance(edge_index, list):
            raise NotImplementedError("list-valued edge_index (edge_type='merge') is not selected by any shipped config")
        if args.device_num != 1:
            n_edge = edge_index.shape[-1] // args.device_num
            edge_index, edge_attr = edge_index[:, :n_edge].contiguous(), edge_attr[:n_edge]
        edge_index = edge_index.to(x.device)
        edge_attr = edge_attr.to(x.device) if args.weighted_edge else None
        static_key = getattr(input_batch, "topology_key", None)
        if edge_attr is not None:
            # one Topology for all layers: the batch is B offset copies of the fold-constant edge list
            # (multiloader.py:687-698) -> single-graph CSR streamed over the B stacked feature blocks
            graph.topology(edge_index, x.shape[0], self_loops=True, edge_weight=edge_attr, static_key=static_key,
                           period=n3)

        feats = []
        mask_col = mask_x.reshape(-1, 1)
        n_layers = len(self.gnn_model)
        if args.node_embedding:
            if (self.input_emb_drop is None and not args.resgnn and args.gnn_name.lower() in ("sage", "rsage")):
                # K13 folded into K7: x0 = x * node_embedding stays factored for the first layer
                x = Fn.RankOne(xs, self.node_embedding)
            else:
                x = Fn.EmbedScale.apply(xs, self.node_embedding)     # [B*N, emb_dim]
                if self.input_emb_drop is not None:
                    x = self.input_emb_drop(x)
        # Activation-backward fusion along a plain layer chain (x_{i+1} = y_i, nothing else reads y_i): the consumer
        # of y_i multiplies its input gradient by LeakyReLU'(y_i) inside its own backward kernel (it has y_i in
        # hand), and layer i takes that gradient as dL/dz -- one 3-tensor elementwise pass per layer saved.
        plain = self.FUSE_ACT_BACKWARD and xs.is_cuda and not args.dense_gnn and not args.resgnn \
            and not args.repeat_mask and (fused or torch.is_grad_enabled())
        slopes = [getattr(l, "grad_fusion_slope", lambda: None)() if plain else None for l in self.gnn_model]
        pool_masks = plain and slopes[-1] is not None and (not (args.value_att_mask and value_mask) or args.merge_mode == 'mult')
        pool_link, layer_links = {}, {}
        for i, layer in enumerate(self.gnn_model):
            if plain and slopes[i] is not None:
                masks = lambda l: getattr(l, "masks_input_grad", lambda: not getattr(l, "relative", True))()
                consumer_masks = pool_masks if i + 1 == n_layers else \
                    (slopes[i + 1] is not None and masks(self.gnn_model[i + 1]))
                producer_masked = i > 0 and slopes[i - 1] is not None and masks(layer)
                # last layer + pool: a dict both Functions see, through which they agree on the layout of the gradient the
                # pool's backward hands to the layer's backward (Fn.SageLayer / Fn.PathwayPool, ``gz_node_major``)
                link = pool_link if (i + 1 == n_layers and consumer_masks) else None
                if (i + 1 != n_layers and self._takes_node_major(self.gnn_model[i + 1], slopes[i + 1])
                        and not self._hooked(layer) and not self._hooked(self.gnn_model[i + 1])):
                    # layer -> layer: the next layer runs transform-first on 32-wide rows; this one may hand it NODE-MAJOR rows
                    link = layer_links[i] = {"want_h1_nm": True}
                layer._mlg_fuse = (slopes[i - 1] if producer_masked else None, bool(consumer_masks), link,
                                   layer_links.get(i - 1))
            y = layer(x, edge_index, edge_attr)
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
                x = x * mask_col
        if args.dense_gnn:
            x = torch.cat(feats, dim=-1)

        vm = None
        if args.value_att_mask and value_mask:
            if args.merge_mode == 'mult':
                # folded into the pool kernel; differentiable: the pool returns dL/dvm when batch.x requires grad
                vm = mask_x.reshape(-1).float().contiguous()
            else:
                x = args.add_coef1 * x + args.add_coef2 * mask_col

        layout = graph.pool_layout(gene_pca_match, raw_indice, n3, 146 * 3,
                                   wrap_negative=not args.pca_match_mask, static_key=static_key)
        # w = learnable_pca_params * info_mask [G, P] (multilevel_gnn.py:222): the mask product and its backward are folded
        # into the pool Function (the projection gradient lands in the parameter's bucket slot)
        x = Fn.PathwayPool.apply(x, self.learnable_pca_params, vm, layout, slopes[-1] if pool_masks else None,
                                 self.info_mask, pool_link if pool_masks else None)   # [B, C, 438, P]
        return x

    @staticmethod
    def _hooked(layer):
        """A forward (pre-)hook sees the layer's input / output rows: they must then be in the reference's graph-major order."""
        mods = [layer, getattr(layer, "gconv", layer)]
        return any(m._forward_hooks or m._forward_pre_hooks for m in mods)

    @staticmethod
    def _takes_node_major(layer, slope):
        """Static part of the layer-to-layer layout hand-shake (Fn.SageLayer): the consumer is a fused, non-relative SAGE layer
        that will run transform-first with 32 output channels (the node-major aggregation kernel's row width)."""
        conv = getattr(layer, "gconv", layer)
        return (slope is not None and Fn.TRANSFORM_FIRST and Fn.H1_NODE_MAJOR and getattr(conv, "relative", True) is False
                and getattr(conv, "out_channels", 0) == 32 and getattr(conv, "in_channels", 0) > 32
                and getattr(conv, "in_channels", 0) % 4 == 0)

    def forward(self, input_batch, x=None, gene_pca_match=None, raw_indice=None, age=None, require_grad=True,
                _loss_args=None, _fused=False):
        with torch.enable_grad() if require_grad else torch.no_grad():
            if x is None:
                age = input_batch.age
            x = self.pool_genes(input_batch, x, gene_pca_match, raw_indice, value_mask=True, fused=_fused)     # [B, C, 438, P]
        return self.post_pool(x, age, require_grad, _loss_args)

    def post_pool(self, x, age, require_grad=True, _loss_args=None):
        """The part of ``forward`` after the gene -> pathway pool: ``x`` the pooled tensor [B, C, 438, P] (as ``pool_genes``
        returns it), ``age`` [B] -> ``(pred, pca_feature)``.  The reshape to [B, C, 146, 3P] and the pathway reorder run under
        the grad mode ``require_grad`` selects, the head under the caller's."""
        args = self.args
        loss_args = _loss_args
        with torch.enable_grad() if require_grad else torch.no_grad():
            x = x.reshape(x.shape[0], x.shape[1], 146, self.pca_dim * 3)
            if args.reorder_pathway and self.reorder_idxs is not None:
                x = x[:, :, self.reorder_idxs.to(x.device), :]

        pca_feature = x
        if self.FUSED_HEAD and self._fused_head_ok(x):
            # head + loss as four kernels (csrc/head.cu): conv1x1+ReLU x2 + max-pool + dropout + flatten + cat(age), then
            # Linear+ReLU+dropout + Linear(->2) + softmax (+ weighted BCE when the trainer passes the target)
            ks = self.pooling.kernel_size if isinstance(self.pooling.kernel_size, tuple) else (self.pooling.kernel_size,) * 2
            a0 = Fn.HeadConvPool.apply(x, self.conv_model[0].weight, self.conv_model[0].bias, self.conv_model[2].weight,
                                       self.conv_model[2].bias, age if args.use_age else None, int(ks[0]), int(ks[1]),
                                       self.drop1.p, self.training)
            y, w = loss_args if loss_args is not None else (None, None)
            pred, bce = Fn.HeadMLP.apply(a0, self.head[0].weight, self.head[0].bias, self.head[3].weight, self.head[3].bias,
                                         self.head[2].p, self.training, y, w)
            self._last_bce = bce if y is not None else None
            return pred, pca_feature
        self._last_bce = None
        layers, i = list(self.conv_model), 0
        while i < len(layers):
            # Conv2d(1x1) + ReLU pairs: the ReLU runs in the GEMM epilogue (forward hooks on either module: unfused)
            fuse = (x.is_cuda and i + 1 < len(layers) and isinstance(layers[i], nn.Conv2d) and layers[i].kernel_size == (1, 1)
                    and type(layers[i + 1]) is nn.ReLU and not layers[i]._forward_hooks and not layers[i + 1]._forward_hooks)
            x = self._conv(layers[i], x, relu=fuse)
            i += 2 if fuse else 1
        pool = self.pooling
        ks = pool.kernel_size if isinstance(pool.kernel_size, tuple) else (pool.kernel_size,) * 2
        if (x.is_cuda and x.dtype == torch.float32 and x.permute(0, 2, 3, 1).is_contiguous()
                and pool.stride in (ks, pool.kernel_size) and pool.padding in (0, (0, 0)) and pool.dilation in (1, (1, 1))
                and not pool.ceil_mode and not pool.return_indices):
            x = Fn.MaxPoolCL.apply(x, int(ks[0]), int(ks[1]))     # channel-last in, NCHW out, no layout copies
        else:
            x = pool(x.contiguous())          # NCHW copy: the library's NHWC max-pool kernels are ~7x slower here
        x = self.drop1(x)
        x = torch.flatten(x, start_dim=1)
        if args.use_age:
            x = torch.cat([x, age[:, None]], dim=-1)
        for mod in self.head:
            # wide first Linear (6913 / 84096 inputs): weight gradient through mlg_xty (cuBLAS picks a slow large-k kernel)
            x = Fn.tall_linear(x, mod, min_rows=1) if (isinstance(mod, nn.Linear) and mod.in_features >= 1024) else mod(x)
        return x, pca_feature

    def predict(self, input_batch):
        """Forward-only evaluation: ``(pred, pca_feature)`` as ``forward`` returns them, in eval semantics (no dropout) whatever
        ``self.training`` and the grad mode, on the kernel route of the training forward -- the factored first layer, node-major
        rows into the transform-first second layer, the fused pool and the fused head -- with no backward state: nothing is
        recorded for autograd and no tensor outlives the call but the two outputs.  Configurations outside the fused chain (dense
        / residual GNN, repeat_mask, hooked layers, unfused heads) run the same generic route as ``forward``.
        ``model(batch)`` under ``torch.no_grad()`` keeps its own (generic) route."""
        was = self.training
        self.train(False)
        try:
            with torch.no_grad():
                return self.forward(input_batch, require_grad=False, _fused=True)
        finally:
            self.train(was)

    def forward_with_loss(self, input_batch, target, weight=None):
        """(pred, pca_feature, bce): ``forward`` plus torch.nn.BCELoss(weight)(pred, target) (train.py:60,118) computed by
        the head kernel that produces ``pred`` (one launch instead of the library's softmax / BCE chain)."""
        pred, feat = self.forward(input_batch, _loss_args=(target, weight))
        bce = self._last_bce
        if bce is None:       # unfused head (hooks, other channel counts, CPU tensors never get here)
            crit = torch.nn.BCELoss(weight=weight) if weight is not None else torch.nn.BCELoss()
            bce = crit(pred.to(torch.float32), target.to(torch.float32))
        self._last_bce = None
        return pred, feat, bce

    FUSED_HEAD = True

    def _fused_head_ok(self, x):
        """The fused head kernels cover the head every shipped config builds: two 1x1 convs 32 -> 32 -> 64 with ReLUs, a
        stride = kernel floor-mode max-pool, Linear/ReLU/Dropout/Linear(->2)/Softmax; no forward hooks on those modules."""
        cm, hd, pool = self.conv_model, self.head, self.pooling
        if not (len(cm) == 4 and isinstance(cm[0], nn.Conv2d) and isinstance(cm[2], nn.Conv2d) and type(cm[1]) is nn.ReLU
                and type(cm[3]) is nn.ReLU and len(hd) == 5 and isinstance(hd[0], nn.Linear) and type(hd[1]) is nn.ReLU
                and isinstance(hd[2], nn.Dropout) and isinstance(hd[3], nn.Linear) and isinstance(hd[4], nn.Softmax)):
            return False
        mods = list(cm) + list(hd) + [pool, self.drop1]
        if any(m._forward_hooks or m._forward_pre_hooks or m._backward_hooks for m in mods):
            return False
        ks = pool.kernel_size if isinstance(pool.kernel_size, tuple) else (pool.kernel_size,) * 2
        if not (pool.stride in (ks, pool.kernel_size) and pool.padding in (0, (0, 0)) and pool.dilation in (1, (1, 1))
                and not pool.ceil_mode and not pool.return_indices):
            return False
        if x.shape[0] > 64 or not Fn.HeadConvPool.supported(x, cm[0], cm[2]):
            return False
        f_in = cm[2].out_channels * (x.shape[2] // ks[0]) * (x.shape[3] // ks[1]) + (1 if self.args.use_age else 0)
        return (hd[0].in_features == f_in and hd[3].out_features == 2 and hd[0].out_features % 32 == 0
                and hd[0].out_features <= 512 and hd[0].bias is not None and hd[3].bias is not None
                and hd[4].dim in (1, -1))

    @staticmethod
    def _conv(layer, x, relu=False):
        """1x1 convolutions run as a matmul over the channel axis: (a) cuDNN's convolution path defaults to TF32
        (torch.backends.cudnn.allow_tf32), which breaks the fp32 rtol-1e-4 parity with the reference; (b) the pooled
        tensor is channel-last in memory (PathwayPool), so [B,C,H,W] -> [B*H*W, C] is a free view and the conv is one
        tall [B*H*W, C] x [C, O] product (3xTF32 tensor-core kernel; weight/bias gradient through mlg_xty instead of
        an 18-way split-K library GEMM)."""
        if isinstance(layer, nn.Conv2d) and layer.kernel_size == (1, 1):
            b, c, hh, ww = x.shape
            x2 = x.permute(0, 2, 3, 1).reshape(-1, c)
            w = layer.weight.view(layer.out_channels, c)
            if x2.is_cuda:
                y2 = Fn.TallLinear.apply(x2, w, layer.bias, relu)
            else:
                y2 = torch.nn.functional.linear(x2, w, layer.bias)
            return y2.view(b, hh, ww, layer.out_channels).permute(0, 3, 1, 2)
        return layer(x)

    # ------------------------------------------------------------------------------------------
    def init_weight(self):
        for m in self.modules():
            if isinstance(m, (nn.Conv2d, nn.Linear)):
                nn.init.xavier_uniform_(m.weight.data)

    def set_pca_params(self, pca_params, mutual_info_mask):
        keep = [i for i in range(len(mutual_info_mask)) if mutual_info_mask[i] > 0]
        self.learnable_pca_params = nn.Parameter(torch.zeros([len(mutual_info_mask), self.pca_dim]),
                                                 requires_grad=not self.args.freeze_pca_weight)
        self.learnable_pca_params.data[keep] = pca_params[:, :self.pca_dim].to(torch.float32)

    def set_pathway_indexs(self, pathway_indexs):
        self.pathway_indexs = pathway_indexs

    def set_info_mask(self, info_mask):
        self.info_mask = nn.Parameter(data=info_mask, requires_grad=False)

    def set_reorder_idxs(self, reorder_idx):
        self.reorder_idxs = torch.tensor(reorder_idx)

    def get_feature_loss(self, pca_feature):
        """-log mean std of pooled features (pca_loss) and the pathway-wise |cos| between projection
        columns (pca_indep_loss, no grad: the reference reads ``.data``), multilevel_gnn.py:329-348 --
        including its loop structure: only the last (i, j) pair of each i is accumulated."""
        loss = 0
        if self.pca_loss:
            flat = pca_feature.reshape(pca_feature.shape[0], -1)
            loss = loss - self.pca_loss_coef * torch.log(torch.mean(torch.std(flat, dim=0)))
        if self.pca_indep_loss:
            dev = self.learnable_pca_params.device
            idx = self.pathway_indexs.to(dev)
            nseg = int(self.pathway_indexs.max()) + 1 if not hasattr(self, "_nseg") else self._nseg
            self._nseg = nseg

            # only the LAST j of every i survives the reference's loop (j = pca_dim - 1): all pairs (i, P-1) at once,
            # one segment sum over [w_i * w_last | w_i^2 | w_last^2] instead of three index_adds per pair
            P = self.pca_dim
            segptr = self._segment_pointers(idx, nseg) if (dev.type == "cuda" and 2 <= P <= 8) else None
            if segptr is not None:
                # genes sorted by pathway: the whole term is ONE launch (mlg_pca_indep_loss) instead of ~14 tiny ones
                from .. import _cabi
                out = torch.empty(1, dtype=torch.float32, device=dev)
                wr = self.learnable_pca_params.data
                mk = self.info_mask.data.reshape(-1)
                wr = wr if (wr.dtype == torch.float32 and wr.is_contiguous()) else wr.float().contiguous()
                mk = mk if (mk.dtype == torch.float32 and mk.is_contiguous()) else mk.float().contiguous()
                with torch.cuda.device(dev):
                    ws = torch.empty(nseg, dtype=torch.float32, device=dev)
                    _cabi.check(_cabi.lib().mlg_pca_indep_loss(_cabi.fptr(wr), _cabi.fptr(mk), _cabi.iptr(segptr), nseg, P,
                                                              _cabi.fptr(out), _cabi.fptr(ws), _cabi.stream_ptr()),
                                "mlg_pca_indep_loss")
                return out[0] if (isinstance(loss, int) and loss == 0) else loss + out[0]
            w = (self.learnable_pca_params * self.info_mask).data     # (the kernel above multiplies the mask in itself)
            if P > 1:
                a, b = w[:, :P - 1], w[:, P - 1:P]
                seg = torch.zeros(nseg, 2 * (P - 1) + 1, device=w.device, dtype=w.dtype).index_add_(
                    0, idx, torch.cat([a * b, a * a, b * b], dim=1))
                mul, ln = seg[:, :P - 1], torch.sqrt(seg[:, P - 1:2 * (P - 1)] * seg[:, 2 * (P - 1):])
                indep = torch.abs(mul / (ln + 1e-7)).mean(dim=0).sum()
                count = P * (P - 1) // 2
            else:
                indep, count = 0, 1
            loss = loss + indep / count
        return loss

    def _segment_pointers(self, idx, nseg):
        """int32 [nseg+1] segment boundaries when ``pathway_indexs`` is sorted (it is for the reference's loaders), else
        None; checked once per index tensor (one host sync, before any graph capture)."""
        key = (idx.data_ptr(), idx._version, tuple(idx.shape), nseg)
        cache = getattr(self, "_segptr_cache", None)
        if cache is None or cache[0] != key:
            ok = idx.numel() > 0 and bool((idx[1:] >= idx[:-1]).all()) and int(idx.min()) >= 0
            ptr = None
            if ok:
                ptr = torch.searchsorted(idx.contiguous(), torch.arange(nseg + 1, device=idx.device, dtype=idx.dtype)).to(torch.int32)
            self._segptr_cache = cache = (key, ptr)
        return cache[1]

    def generate_mutual_mask(self, *a, **k):
        raise NotImplementedError("sklearn mutual-information data prep is out of scope (SURVEY.md section 2 row 7)")
