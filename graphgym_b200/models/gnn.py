"""The callers either side of the message-passing stage, as GraphGym stacks them (ref: graphgym/models/gnn.py:21-174,
graphgym/models/head.py:15-43): ``GNNPreMP`` (linear layers), the stage ``stage_dict[cfg.gnn.stage_type]`` —
``GNNStackStage`` (cfg.gnn.layers_mp GeneralLayers of cfg.gnn.layer_type) or ``GNNSkipStage`` (skip blocks of
cfg.gnn.skip_every layers, 'skipsum' / 'skipconcat'), L2-normalised at the end of the stage when cfg.gnn.l2norm — and
``GNNNodeHead`` (MLP on the rows ``node_id_index`` selects).  Kept thin: everything heavy is the layers' gg_* path; the
stage's final L2 normalisation is folded into the last layer's (stack) or the last block's (skip) fused post-op pass
instead of running as a separate F.normalize.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from graphgym_b200 import functional as F_
from graphgym_b200 import ops
from graphgym_b200.config import cfg
from graphgym_b200.models.layer import _ACT, _FUSED_ACT, TFG_ALIASES, GeneralLayer


class GNNStackStage(nn.Module):
    """ref: gnn.py:65-81 — ``layer{i}`` children, then F.normalize(p=2, dim=-1) if cfg.gnn.l2norm."""

    def __init__(self, dim_in, dim_out, num_layers, layer_type=None):
        super().__init__()
        name = layer_type or cfg.gnn.layer_type
        name = TFG_ALIASES.get(name, name)
        for i in range(num_layers):
            d_in = dim_in if i == 0 else dim_out
            last = i == num_layers - 1
            self.add_module('layer{}'.format(i), GeneralLayer(name, d_in, dim_out, has_act=True,
                                                              has_l2norm=bool(cfg.gnn.l2norm) and last))
        self.dim_out = dim_out

    def forward(self, batch):
        for layer in self.children():
            batch = layer(batch)
        return batch


class GNNSkipBlock(nn.Module):
    """ref: gnn.py GNNSkipBlock — ``f`` = ``num_layers`` GeneralLayers (the last one without activation: BN and dropout
    only), ``act`` = the stage activation, then act(x + f(x)) ('skipsum', needs dim_in == dim_out) or
    act(cat([x, f(x)], 1)) ('skipconcat': the carried columns are activated too); ``has_l2norm``: the stage's final
    F.normalize, applied here when this is the stage's last block.

    On CUDA fp32 input with an activation of the fused set and no active dropout, the last layer runs its conv only and
    its BatchNorm, the skip connection, the activation and the L2 run as ONE epilogue (``functional.skip_post_ops``);
    otherwise (PReLU / ELU / SELU, dropout > 0 while training, cfg.b200.fused_postops off) the modules run one by one."""

    def __init__(self, dim_in, dim_out, num_layers, layer_type=None, has_l2norm=False):
        super().__init__()
        self.stage_type = cfg.gnn.stage_type
        if self.stage_type not in ('skipsum', 'skipconcat'):
            raise ValueError("cfg.gnn.stage_type must be 'skipsum' or 'skipconcat' for a skip block, got {!r}".format(
                self.stage_type))
        if self.stage_type == 'skipsum' and dim_in != dim_out:
            raise ValueError('a skipsum block needs dim_in == dim_out, got {} and {}'.format(dim_in, dim_out))
        name = layer_type or cfg.gnn.layer_type
        name = TFG_ALIASES.get(name, name)
        self.f = nn.Sequential(*[GeneralLayer(name, dim_in if i == 0 else dim_out, dim_out,
                                              has_act=i < num_layers - 1) for i in range(num_layers)])
        self.act = _ACT[cfg.gnn.act]()
        self.has_l2norm = bool(has_l2norm)
        self._act = _FUSED_ACT.get(cfg.gnn.act)
        self._drop_p = cfg.gnn.dropout
        self._mode = ops.SKIP_SUM if self.stage_type == 'skipsum' else ops.SKIP_PREFIX

    def forward(self, batch):
        x = batch.node_feature
        fused = (x.is_cuda and x.dim() == 2 and x.dtype == torch.float32 and self._act is not None
                 and not (self._drop_p > 0 and self.training) and cfg.b200.fused_postops)
        if fused:
            for layer in self.f[:-1]:
                batch = layer(batch)
            last = self.f[-1]
            batch = last.layer(batch)
            bn = last.post_layer[0] if last._has_bn else None
            batch.node_feature = F_.skip_post_ops(batch.node_feature, x, self._mode, bn, self.training, self._act[0],
                                                  self._act[1], self.has_l2norm)
            return batch
        h = self.f(batch).node_feature
        h = x + h if self._mode == ops.SKIP_SUM else torch.cat([x, h], 1)
        h = self.act(h)
        if self.has_l2norm:
            h = F.normalize(h, p=2, dim=-1)
        batch.node_feature = h
        return batch


class GNNSkipStage(nn.Module):
    """ref: gnn.py GNNSkipStage — ``block{i}`` children, num_layers // cfg.gnn.skip_every of them; block i takes dim_in
    (i = 0), then dim_out ('skipsum') or dim_in + i * dim_out ('skipconcat'); F.normalize(p=2, dim=-1) at the end if
    cfg.gnn.l2norm (folded into the last block)."""

    def __init__(self, dim_in, dim_out, num_layers, layer_type=None):
        super().__init__()
        k = int(cfg.gnn.skip_every)
        if k < 1 or num_layers % k != 0:
            raise ValueError('cfg.gnn.layers_mp = {} must be a multiple of cfg.gnn.skip_every = {}'.format(num_layers, k))
        concat = cfg.gnn.stage_type == 'skipconcat'
        blocks = num_layers // k
        for i in range(blocks):
            d_in = dim_in if i == 0 else (dim_in + i * dim_out if concat else dim_out)
            self.add_module('block{}'.format(i), GNNSkipBlock(d_in, dim_out, k, layer_type,
                                                              has_l2norm=bool(cfg.gnn.l2norm) and i == blocks - 1))
        self.dim_out = dim_in + blocks * dim_out if concat else dim_out

    def forward(self, batch):
        for block in self.children():
            batch = block(batch)
        return batch


stage_dict = {'stack': GNNStackStage, 'skipsum': GNNSkipStage, 'skipconcat': GNNSkipStage}


class _Linear(nn.Module):
    """``linear`` of the reference's layer_dict (ref: models/layer.py:73-86) on the gg GEMM."""

    def __init__(self, dim_in, dim_out, bias=False, **kwargs):
        super().__init__()
        self.model = nn.Linear(dim_in, dim_out, bias=bias)

    def forward(self, batch):
        if isinstance(batch, torch.Tensor):
            return F_.linear(batch, self.model.weight, self.model.bias)
        batch.node_feature = F_.linear(batch.node_feature, self.model.weight, self.model.bias)
        return batch


class GNNPreMP(nn.Module):
    """ref: gnn.py:40-62 (GeneralMultiLayer('linear', ...)): Linear -> BN -> act per layer, fused post-ops."""

    def __init__(self, dim_in, dim_out, num_layers=1):
        super().__init__()
        from graphgym_b200.models import layer as L
        L.layer_dict.setdefault('linear', _Linear)
        for i in range(num_layers):
            self.add_module('Layer_{}'.format(i), GeneralLayer('linear', dim_in if i == 0 else dim_out, dim_out, True))
        self.dim_out = dim_out

    def forward(self, batch):
        for layer in self.children():
            batch = layer(batch)
        return batch


class GNNNodeHead(nn.Module):
    """ref: head.py:15-43 — the prediction MLP on the rows ``node_id_index`` selects (the centre copies of the ego-nets)
    or on all rows; returns (pred, label)."""

    def __init__(self, dim_in, dim_out):
        super().__init__()
        self.layer_post_mp = nn.Linear(dim_in, dim_out, bias=True)

    def forward(self, batch):
        h = batch.node_feature
        ids = getattr(batch, 'node_id_index', None)
        if ids is not None:
            h = F_.gather_rows(h, ids)
        pred = F_.linear(h, self.layer_post_mp.weight, self.layer_post_mp.bias)
        return pred, getattr(batch, 'node_label', None)


class GNN(nn.Module):
    """ref: gnn.py:139-174 — pre_mp -> mp stage (``stage_dict[cfg.gnn.stage_type]``) -> post_mp head on the stage's
    dim_out, dimensions from cfg.gnn."""

    def __init__(self, dim_in, dim_out):
        super().__init__()
        stage = stage_dict.get(cfg.gnn.stage_type)
        if stage is None:
            raise ValueError('cfg.gnn.stage_type = {!r}: one of {}'.format(cfg.gnn.stage_type, sorted(stage_dict)))
        d = cfg.gnn.dim_inner
        if cfg.gnn.layers_pre_mp > 0:
            self.pre_mp = GNNPreMP(dim_in, d, cfg.gnn.layers_pre_mp)
            dim_in = d
        if cfg.gnn.layers_mp > 0:
            self.mp = stage(dim_in, d, cfg.gnn.layers_mp)
            dim_in = self.mp.dim_out
        self.post_mp = GNNNodeHead(dim_in, dim_out)

    def forward(self, batch):
        for module in self.children():
            batch = module(batch)
        return batch
