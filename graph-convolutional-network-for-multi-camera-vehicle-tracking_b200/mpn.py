"""Drop-in ``MOTMPNet`` for the reference's tracklet-graph message-passing network.

Same constructor (``MOTMPNet(model_params, bb_encoder=None, arch)``, models/mpn.py:154), same ``state_dict``
keys and shapes (so ``utils.load_pretrained_weights`` works unchanged, utils.py:482-531) and the same
``forward(data) -> ({'classified_edges': [...]}, latent_node_feats)`` contract (models/mpn.py:250-299).
The parameters live in ordinary ``nn.Linear`` / ``nn.BatchNorm1d`` modules arranged exactly as the reference's
``nn.Sequential`` numbers them (models/mlp.py:11-30); the computation is done by libmpn_b200's sm_100a kernels.
There is no PyTorch/CPU fallback for ``forward``.
"""
import ctypes as C

import torch
from torch import nn

from . import _lib
from .graph import _on_device, current_stream_ptr, graph_for, node_features, workspace

USE_TENSOR_CORES = True


class _GraphedForward:
    """One captured CUDA graph of ``mpn_forward`` for a fixed (N, E, weights) signature.

    Inputs are staged into static buffers (skipped when the caller passes the same tensors again), the graph is
    replayed with a single launch, outputs are cloned so the caller still receives fresh tensors like the reference.
    """

    def __init__(self, W, g, x, x_kind, ea, L, n_cls, n_out, fused):
        from .graph import TrackletGraph
        dev = x.device
        self.W, self.L, self.n_cls = W, L, n_cls
        self.x, self.ea = torch.empty_like(x), torch.empty_like(ea)      # x staged in its own dtype
        # static graph tables with the same sizes as the caller's
        self.g = object.__new__(TrackletGraph)
        for name in ("device", "n_cols", "n_nodes", "row_offset", "n_edges", "chunk", "max_tasks"):
            setattr(self.g, name, getattr(g, name))
        self.g.perm = None
        self.tables = ("rowptr", "col", "taskptr", "task_row", "n_tasks")
        for name in self.tables:
            setattr(self.g, name, torch.empty_like(getattr(g, name)))
        self.g.n_graphs, self.g.node_gid, self.g.graph_nptr, self.g.max_graph_nodes = g.n_graphs, None, None, g.max_graph_nodes
        if g.n_graphs > 1:
            self.tables = self.tables + ("node_gid", "graph_nptr")
            self.g.node_gid, self.g.graph_nptr = torch.empty_like(g.node_gid), torch.empty_like(g.graph_nptr)
        self.g.struct = _lib.MpnGraph(g.n_nodes, g.n_cols, g.row_offset, g.chunk, g.n_edges, g.max_tasks, 0,
                                      self.g.rowptr.data_ptr(), self.g.col.data_ptr(), self.g.taskptr.data_ptr(),
                                      self.g.task_row.data_ptr(), self.g.n_tasks.data_ptr(), g.n_graphs, g.max_graph_nodes,
                                      self.g.node_gid.data_ptr() if g.n_graphs > 1 else None,
                                      self.g.graph_nptr.data_ptr() if g.n_graphs > 1 else None)
        self.logits = torch.empty(n_out, g.n_edges, 2, dtype=torch.float32, device=dev)
        self.h = torch.empty(g.n_nodes, _lib.MPN_DH, dtype=torch.float32, device=dev)
        self.pred = torch.empty(g.n_edges, dtype=torch.uint8, device=dev) if fused else None
        self.prob1 = torch.empty(g.n_edges, dtype=torch.float32, device=dev) if fused else None
        lib = _lib.lib()
        need = lib.mpn_forward_workspace_bytes(self.g.ref, C.byref(W), L)
        self.ws = torch.empty(need + 4096, dtype=torch.uint8, device=dev)      # private: lives as long as the graph
        self._last = None
        self._stage(g, x, ea)

        def launch():
            _lib.check(lib.mpn_forward_x(self.g.ref, C.byref(W), self.x.data_ptr(), x_kind, self.ea.data_ptr(), L, n_cls,
                                         self.logits.data_ptr(), self.h.data_ptr(),
                                         self.pred.data_ptr() if fused else None, self.prob1.data_ptr() if fused else None,
                                         int(bool(USE_TENSOR_CORES)), self.ws.data_ptr(), self.ws.numel(),
                                         current_stream_ptr(dev)))
        with torch.cuda.device(dev):
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):                                       # warm-up outside capture (lazy inits)
                launch()
            torch.cuda.current_stream(dev).wait_stream(side)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                launch()

    def _stage(self, g, x, ea):
        # the graph tables are immutable once built: identity (held through a weak reference) is enough.  The features are
        # ALWAYS copied: tensor identity + _version would miss writes through .data or by a foreign kernel, and at most 2^21
        # edges are staged here (a few microseconds)
        lg = self._last() if self._last is not None else None
        if lg is not g:
            for name in self.tables:
                getattr(self.g, name).copy_(getattr(g, name), non_blocking=True)
            import weakref
            self._last = weakref.ref(g)
        self.x.copy_(x, non_blocking=True)
        self.ea.copy_(ea, non_blocking=True)

    def run(self, g, x, ea):
        self._stage(g, x, ea)
        self.graph.replay()
        return (self.logits.clone(), self.h.clone(), self.pred.clone() if self.pred is not None else None,
                self.prob1.clone() if self.prob1 is not None else None)


class MLP(nn.Module):
    """Parameter container with the reference layout: [Linear, BatchNorm1d, ReLU, Dropout] per hidden width
    (BN/ReLU/Dropout omitted for width 1; bare Linear stack for classifiers) — models/mlp.py:4-33."""

    def __init__(self, input_dim, fc_dims, dropout_p=0.4, use_batchnorm=False, is_classifier=False):
        super().__init__()
        assert isinstance(fc_dims, (list, tuple)), \
            'fc_dims must be either a list or a tuple, but got {}'.format(type(fc_dims))
        mods, self.blocks = [], []
        for width in fc_dims:
            lin_pos, bn_pos = len(mods), None
            mods.append(nn.Linear(input_dim, width))
            if not is_classifier and width != 1:
                if use_batchnorm:
                    bn_pos = len(mods)
                    mods.append(nn.BatchNorm1d(width, track_running_stats=False))
                mods.append(nn.ReLU(inplace=True))
                if dropout_p is not None:
                    mods.append(nn.Dropout(p=dropout_p))
            self.blocks.append((lin_pos, bn_pos))
            input_dim = width
        self.fc_layers = nn.Sequential(*mods)

    def forward(self, input):
        raise RuntimeError("the B200 MLP modules only hold parameters; call MOTMPNet.forward (CUDA kernels)")


class MLPGraphIndependent(nn.Module):
    """Encoder / classifier container (models/mpn.py:103-142)."""

    def __init__(self, edge_in_dim=None, node_in_dim=None, edge_out_dim=None, node_out_dim=None, node_fc_dims=None,
                 edge_fc_dims=None, dropout_p=None, use_batchnorm=None, is_classifier=False):
        super().__init__()
        self.node_mlp = None if node_in_dim is None else MLP(node_in_dim, list(node_fc_dims) + [node_out_dim],
                                                             dropout_p, use_batchnorm, is_classifier)
        self.edge_mlp = None if edge_in_dim is None else MLP(edge_in_dim, list(edge_fc_dims) + [edge_out_dim],
                                                             dropout_p, use_batchnorm, is_classifier)


class EdgeModel(nn.Module):
    def __init__(self, edge_mlp):
        super().__init__()
        self.edge_mlp = edge_mlp


class NodeModel(nn.Module):
    def __init__(self, node_mlp, node_agg_fn):
        super().__init__()
        self.node_mlp = node_mlp
        self.node_agg_fn = node_agg_fn


class MetaLayer(nn.Module):
    def __init__(self, edge_model=None, node_model=None):
        super().__init__()
        self.edge_model = edge_model
        self.node_model = node_model


def _unsupported(what):
    return NotImplementedError("libmpn_b200 does not implement %s (supported family: the shipped configuration "
                               "config/config_training.yaml:68-111 with any node-encoder widths, any num_enc_steps / "
                               "num_class_steps); there is no PyTorch fallback" % what)


class MOTMPNet(nn.Module):
    def __init__(self, model_params, bb_encoder=None, arch=None):
        super().__init__()
        self.node_cnn = bb_encoder
        self.model_params = model_params
        # the reference merges the node-encoder dict into the edge-encoder dict in place (models/mpn.py:167-170)
        edges_params = model_params['encoder_feats_dict']['edges']
        nodes_params = model_params['encoder_feats_dict']['nodes'][arch]
        edges_params.update(nodes_params)
        enc = edges_params
        cls = model_params['classifier_feats_dict']
        self.encoder = MLPGraphIndependent(**enc)
        self.classifier = MLPGraphIndependent(**cls)

        agg = model_params['node_agg_fn']
        assert agg.lower() in ('mean', 'max', 'sum'), "node_agg_fn can only be 'max', 'mean' or 'sum'."
        self.reattach_initial_nodes = model_params['reattach_initial_nodes']
        self.reattach_initial_edges = model_params['reattach_initial_edges']
        edge_factor = 2 if self.reattach_initial_edges else 1
        node_factor = 2 if self.reattach_initial_nodes else 1
        edge_in = node_factor * 2 * enc['node_out_dim'] + edge_factor * enc['edge_out_dim']
        node_in = node_factor * enc['node_out_dim'] + enc['edge_out_dim']
        em, nm = model_params['edge_model_feats_dict'], model_params['node_model_feats_dict']
        self.MPNet = MetaLayer(
            edge_model=EdgeModel(MLP(edge_in, em['fc_dims'], em['dropout_p'], em['use_batchnorm'])),
            node_model=NodeModel(MLP(node_in, nm['fc_dims'], nm['dropout_p'], nm['use_batchnorm']), agg))
        self.num_enc_steps = model_params['num_enc_steps']
        self.num_class_steps = model_params['num_class_steps']

        # ---- what the kernels support; checked once here so forward() fails early and loudly ----
        self._node_agg = {'sum': _lib.AGG_SUM, 'mean': _lib.AGG_MEAN, 'max': _lib.AGG_MAX}[agg.lower()]    # models/mpn.py:196-202
        if not (enc['edge_in_dim'] == 2 and list(enc['edge_fc_dims']) == [4] and enc['edge_out_dim'] == 4):
            raise _unsupported("an edge encoder other than 2->[4]->4")
        if enc['node_out_dim'] != _lib.MPN_DH or len(enc['node_fc_dims']) + 1 > _lib.MPN_MAX_NODE_LAYERS:
            raise _unsupported("node_out_dim != 32 or more than 8 node-encoder layers")
        if not (enc['use_batchnorm'] and em['use_batchnorm'] and nm['use_batchnorm']):
            raise _unsupported("use_batchnorm=False")
        if list(em['fc_dims']) != [4] or list(nm['fc_dims']) != [32]:
            raise _unsupported("edge_model fc_dims != [4] or node_model fc_dims != [32]")
        if not (cls['edge_in_dim'] == 4 and list(cls['edge_fc_dims']) == [] and cls['edge_out_dim'] == 2
                and cls.get('is_classifier', False)):
            raise _unsupported("a classifier other than Linear 4->2")
        if any(w == 1 for w in list(enc['node_fc_dims'])):
            raise _unsupported("node encoder widths of 1")
        self._packed = None          # (version key, small block tensor, MpnWeights struct, keepalive list)
        # small graphs are launch-bound (~30 dependent kernels): replay the forward as one CUDA graph
        self.use_cuda_graph = True
        self.cuda_graph_max_edges = 1 << 21
        self._graphs = {}            # (device, N, E, D, x dtype, L, n_cls, fused, weights key) -> _GraphedForward
        self.fuse_decisions = False  # when True forward also stores self.last_pred (uint8) / self.last_prob1 (fp32)
        self.last_pred = self.last_prob1 = None

    # ------------------------------------------------------------------------------------------
    def invalidate_weight_cache(self):
        """The packed weights (and their tensor-core planes) are cached and rebuilt when a parameter's data pointer or version
        counter changes: ``load_state_dict``, ``.to()``, in-place ops on the Parameter itself.  Call this after anything those
        two do not see: a Parameter OBJECT replaced (``module.weight = nn.Parameter(...)``), writes through ``p.data`` (``.data``
        has its own version counter) or by a foreign kernel."""
        self.__dict__.pop("_param_list", None)
        self._packed = None

    def _weights(self, device):
        params = self.__dict__.get("_param_list")          # Parameter objects keep their identity across .to() / load_state_dict
        if params is None:                                 # (walking the module tree costs ~40 us per call)
            params = self.__dict__["_param_list"] = list(self.parameters())
        key = (device,) + tuple([(p.data_ptr(), p._version) for p in params])
        if self._packed is not None and self._packed[0] == key:
            return self._packed[2]
        for p in params:
            if p.device != device or p.dtype != torch.float32:
                raise RuntimeError("all MOTMPNet parameters must be fp32 on %s (got %s %s)" % (device, p.dtype, p.device))
        W = _lib.MpnWeights()
        W.node_agg = self._node_agg
        keep = []
        nmlp = self.encoder.node_mlp
        W.n_node_layers = len(nmlp.blocks)
        for i, (lin, bn) in enumerate(nmlp.blocks):
            l, b = nmlp.fc_layers[lin], nmlp.fc_layers[bn]
            if i == 0:
                W.node_dims[0] = l.in_features
            W.node_dims[i + 1] = l.out_features
            ts = [l.weight.detach().contiguous(), l.bias.detach().contiguous(), b.weight.detach().contiguous(),
                  b.bias.detach().contiguous()]
            keep += ts
            W.node_w[i], W.node_b[i], W.node_gamma[i], W.node_beta[i] = (t.data_ptr() for t in ts)
            if ts[0].numel() % 4 == 0:
                # TF32 hi/lo planes of the weight, made once per weight version (operands of the 3xTF32 GEMM)
                hi, lo = torch.empty_like(ts[0]), torch.empty_like(ts[0])
                with torch.cuda.device(device):
                    _lib.check(_lib.lib().mpn_split_tf32(ts[0].data_ptr(), ts[0].numel(), hi.data_ptr(), lo.data_ptr(),
                                                         current_stream_ptr(device)))
                keep += [hi, lo]
                W.node_w_hi[i], W.node_w_lo[i] = hi.data_ptr(), lo.data_ptr()
                if l.in_features % 8 == 0:
                    # fp16 planes of weight * 2^k (operands of the 3xFP16 GEMM: twice the tensor-pipe rate of TF32, same 22 bits)
                    hi16 = torch.empty(ts[0].shape, dtype=torch.float16, device=device)
                    lo16 = torch.empty_like(hi16)
                    scale = C.c_float(0.0)
                    with torch.cuda.device(device):
                        _lib.check(_lib.lib().mpn_split_f16(ts[0].data_ptr(), ts[0].numel(), float(ts[0].abs().max()),
                                                            hi16.data_ptr(), lo16.data_ptr(), C.byref(scale),
                                                            current_stream_ptr(device)))
                    keep += [hi16, lo16]
                    W.node_w_hi16[i], W.node_w_lo16[i], W.node_w_scale16[i] = hi16.data_ptr(), lo16.data_ptr(), scale.value
            # bound of the next layer's input: |relu(BN(y))| <= max|beta| + max|gamma| * sqrt(M - 1)
            W.node_bn_gmax[i], W.node_bn_bmax[i] = float(ts[2].abs().max()), float(ts[3].abs().max())
        small = torch.zeros(_lib.W_SMALL_FLOATS, dtype=torch.float32, device=device)

        def put(off, t):
            small[off:off + t.numel()] = t.detach().reshape(-1)

        e = self.encoder.edge_mlp
        (l1, b1), (l2, b2) = e.blocks
        put(_lib.W_ENC1_W, e.fc_layers[l1].weight); put(_lib.W_ENC1_B, e.fc_layers[l1].bias)
        put(_lib.W_ENC1_G, e.fc_layers[b1].weight); put(_lib.W_ENC1_BETA, e.fc_layers[b1].bias)
        put(_lib.W_ENC2_W, e.fc_layers[l2].weight); put(_lib.W_ENC2_B, e.fc_layers[l2].bias)
        put(_lib.W_ENC2_G, e.fc_layers[b2].weight); put(_lib.W_ENC2_BETA, e.fc_layers[b2].bias)
        # MPNet weights.  With reattach_initial_nodes / _edges (models/mpn.py:207-215, 283-287) the inputs are
        # [h0_row | h_row | h0_col | h_col | e0 | e] (edge MLP) and [h0_row | h_row | e'] (node MLP), initial encodings first:
        # the columns of the current features go to the [4,68] / [32,36] blocks, those of the initial encodings to the *_W0 blocks.
        re_n, re_e = bool(self.reattach_initial_nodes), bool(self.reattach_initial_edges)
        W.reattach_nodes, W.reattach_edges = int(re_n), int(re_e)
        D, De = _lib.MPN_DH, 4
        m = self.MPNet.edge_model.edge_mlp
        (l, b), = m.blocks
        we = m.fc_layers[l].weight.detach()
        nb = 2 if re_n else 1
        h_row, h_col = we[:, (nb - 1) * D:nb * D], we[:, (2 * nb - 1) * D:2 * nb * D]
        e_cur = we[:, 2 * nb * D + (De if re_e else 0):2 * nb * D + (2 * De if re_e else De)]
        put(_lib.W_EDGE_W, torch.cat([h_row, h_col, e_cur], dim=1).contiguous())
        zeros_d, zeros_e = we.new_zeros(we.shape[0], D), we.new_zeros(we.shape[0], De)
        put(_lib.W_EDGE_W0, torch.cat([we[:, 0:D] if re_n else zeros_d, we[:, 2 * D:3 * D] if re_n else zeros_d,
                                       we[:, 2 * nb * D:2 * nb * D + De] if re_e else zeros_e], dim=1).contiguous())
        put(_lib.W_EDGE_B, m.fc_layers[l].bias)
        put(_lib.W_EDGE_G, m.fc_layers[b].weight); put(_lib.W_EDGE_BETA, m.fc_layers[b].bias)
        m = self.MPNet.node_model.node_mlp
        (l, b), = m.blocks
        wn = m.fc_layers[l].weight.detach()
        put(_lib.W_NODE_W, torch.cat([wn[:, (nb - 1) * D:nb * D], wn[:, nb * D:nb * D + De]], dim=1).contiguous())
        put(_lib.W_NODE_W0, (wn[:, 0:D] if re_n else wn.new_zeros(wn.shape[0], D)).contiguous())
        put(_lib.W_NODE_B, m.fc_layers[l].bias)
        put(_lib.W_NODE_G, m.fc_layers[b].weight); put(_lib.W_NODE_BETA, m.fc_layers[b].bias)
        c = self.classifier.edge_mlp
        (l, _), = c.blocks
        put(_lib.W_CLS_W, c.fc_layers[l].weight); put(_lib.W_CLS_B, c.fc_layers[l].bias)
        W.small = small.data_ptr()
        self._packed = (key, small, W, keep)
        return W

    # ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, data):
        """data.x [N,D] fp32 (or fp16 / bf16: read in place, every output equals the one on ``data.x.float()``),
        data.edge_index [2,E] int64, data.edge_attr [E,2] fp32, all on one CUDA device.
        Returns ({'classified_edges': [logits [E,2], ...]}, latent_node_feats [N,32]) as models/mpn.py:299.

        Extension: when ``data.edge_attr`` is None (or absent) the initial edge features of inference.py:453-456 are computed
        here from ``data.x`` — in the same call, so that the node encoder overlaps them on a side stream — and stored back into
        ``data.edge_attr`` (same values as ``edge_features(data.x, data.edge_index)``)."""
        x, edge_attr = data.x, getattr(data, "edge_attr", None)
        # data.mpn_graph: tables built on the device by TrackletGraph.from_cameras (no int64 edge_index needed)
        pre = getattr(data, "mpn_graph", None)
        edge_index = None if pre is not None else data.edge_index
        if not (x.is_cuda and (edge_attr is None or edge_attr.is_cuda) and (edge_index is None or edge_index.is_cuda)):
            raise RuntimeError("MOTMPNet.forward needs CUDA tensors: the B200 path has no CPU fallback")
        if self.training:
            raise _unsupported("training mode (dropout active / autograd); call .eval() as main.py:98 does")
        dev = x.device
        x, x_kind = node_features(x)
        g = pre if pre is not None else graph_for(data, edge_index, x.shape[0])
        W = self._weights(dev)
        make_features = edge_attr is None
        fused_features = (make_features and g.n_graphs <= 1 and g.n_edges > 0 and
                          not (self.use_cuda_graph and g.n_edges <= self.cuda_graph_max_edges))
        if make_features and not fused_features:          # small graphs (CUDA-graph replay), batched graphs: two calls
            from .edge_features import edge_features
            edge_attr = edge_features(x, None, graph=g)
            if g.perm is not None:
                edge_attr = edge_attr[g.perm]             # (edge_features returned the caller's order)
            ea = edge_attr.contiguous()
        elif fused_features:
            ea = torch.empty(g.n_edges, 2, dtype=torch.float32, device=dev)          # filled by the fused call, graph edge order
        else:
            ea = edge_attr.contiguous().float()
            if g.perm is not None:
                ea = ea[g.perm].contiguous()
        if x.shape[1] != W.node_dims[0]:
            raise ValueError("data.x has %d features, the node encoder expects %d" % (x.shape[1], W.node_dims[0]))
        if ea.shape != (g.n_edges, 2):
            raise ValueError("data.edge_attr must be [E,2]")
        L, n_cls = int(self.num_enc_steps), int(self.num_class_steps)
        if L > 0:
            n_cls = min(n_cls, L)         # first_class_step <= 0 classifies every step: L outputs (models/mpn.py:281,290)
        n_out = 1 if L == 0 else n_cls
        fused = bool(self.fuse_decisions) and n_out > 0
        if self.use_cuda_graph and g.n_edges <= self.cuda_graph_max_edges and g.n_edges > 1:
            key = (dev.index, g.n_nodes, g.n_edges, g.n_graphs, g.chunk, g.max_tasks, g.max_graph_nodes, x.shape[1], x.dtype, L,
                   n_cls, bool(self.fuse_decisions), self._packed[0])
            ent = self._graphs.get(key)
            if ent is None:
                if len(self._graphs) >= 8:
                    self._graphs.pop(next(iter(self._graphs)))
                ent = self._graphs[key] = _GraphedForward(W, g, x, x_kind, ea, L, n_cls, max(n_out, 1), fused)
            logits, h, pred, prob1 = ent.run(g, x, ea)
        else:
            logits = torch.empty(max(n_out, 1), g.n_edges, 2, dtype=torch.float32, device=dev)
            h = torch.empty(g.n_nodes, _lib.MPN_DH, dtype=torch.float32, device=dev)
            pred = torch.empty(g.n_edges, dtype=torch.uint8, device=dev) if fused else None
            prob1 = torch.empty(g.n_edges, dtype=torch.float32, device=dev) if fused else None
            lib = _lib.lib()
            need = lib.mpn_forward_workspace_bytes(g.ref, C.byref(W), L)
            ws = workspace("forward", dev, need)
            with _on_device(dev):
                if fused_features:
                    ef_ws = workspace("edge_features", dev, lib.mpn_edge_features_workspace_bytes(g.ref, x.shape[1]))
                    _lib.check(lib.mpn_forward_with_edge_features_x(
                        g.ref, C.byref(W), x.data_ptr(), x_kind, ea.data_ptr(), L, n_cls, logits.data_ptr(), h.data_ptr(),
                        pred.data_ptr() if pred is not None else None, prob1.data_ptr() if prob1 is not None else None,
                        int(bool(USE_TENSOR_CORES)), ws.data_ptr(), ws.numel(), ef_ws.data_ptr(), ef_ws.numel(),
                        current_stream_ptr(dev)))
                else:
                    _lib.check(lib.mpn_forward_x(g.ref, C.byref(W), x.data_ptr(), x_kind, ea.data_ptr(), L, n_cls,
                                                 logits.data_ptr(), h.data_ptr(), pred.data_ptr() if pred is not None else None,
                                                 prob1.data_ptr() if prob1 is not None else None, int(bool(USE_TENSOR_CORES)),
                                                 ws.data_ptr(), ws.numel(), current_stream_ptr(dev)))
        if g.perm is not None:                       # back to the caller's edge order
            inv = torch.empty_like(logits)
            inv[:, g.perm] = logits
            logits = inv
            if pred is not None:
                p2, q2 = torch.empty_like(pred), torch.empty_like(prob1)
                p2[g.perm], q2[g.perm] = pred, prob1
                pred, prob1 = p2, q2
        if make_features:                                 # hand the features back in the caller's edge order
            out_ea = ea
            if g.perm is not None:
                out_ea = torch.empty_like(ea)
                out_ea[g.perm] = ea
            try:
                data.edge_attr = out_ea
            except Exception:
                pass
        self.last_pred, self.last_prob1 = pred, prob1
        return {'classified_edges': [logits[i] for i in range(n_out)]}, h
