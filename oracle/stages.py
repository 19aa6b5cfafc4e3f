"""GraphGym's skip stages (TEST INFRASTRUCTURE ONLY — see oracle/__init__.py), over the oracle layers.

ref: graphgym/models/gnn.py ``GNNSkipBlock`` / ``GNNSkipStage`` / ``stage_dict``:
  block    f = k GeneralLayers: conv -> BatchNorm1d (batch statistics) -> activation, the LAST layer without its
           activation; then  skipsum:    out = act(x + f(x))            (the block needs d_in == dim_out)
                             skipconcat: out = act(cat([x, f(x)], 1))   (the carried x columns are activated again)
  stage    num_layers // skip_every blocks; block i takes dim_in (i = 0), then dim_out (skipsum) or dim_in + i dim_out
           (skipconcat); F.normalize(p=2, dim=-1) after the last block when cfg.gnn.l2norm.

Every activation takes an optional ``gate`` (a bool tensor, True = the positive branch) that replaces its own choice, so
that gradients can be compared under the branches another implementation took (the pattern of ``max_agg``'s ``arg``);
``tap`` collects the pre-activations for the caller's near-tie check.

  activation   relu / leaky relu / prelu with an optional gate
  skip_block   one block over caller-supplied convolutions (e.g. oracle.max_agg.general_conv, oracle.layers.*)
  skip_stage   the blocks, then the stage L2
"""
import torch
import torch.nn.functional as F


def activation(h, act, gate=None):
    """``act``: ('relu',), ('lrelu', slope) or ('prelu', weight [1] or [F]); ``gate``: bool tensor shaped like h, or None
    for the activation's own choice (h > 0)."""
    if gate is None:
        gate = h > 0
    kind = act[0]
    if kind == 'relu':
        neg = torch.zeros_like(h)
    elif kind == 'lrelu':
        neg = h * float(act[1])
    elif kind == 'prelu':
        neg = h * act[1]
    else:
        raise ValueError('activation {!r}'.format(kind))
    return torch.where(gate, h, neg)


def batch_norm(h, bn, eps=1e-5):
    """BatchNorm1d with batch statistics; ``bn`` = (weight, bias) or None (no BN layer)."""
    if bn is None:
        return h
    return F.batch_norm(h, None, None, bn[0], bn[1], True, 0.0, eps)


def skip_block(x, convs, bns, mode, act, gates=None, tap=None, eps=1e-5):
    """One GNNSkipBlock.  ``convs``: k callables h -> conv(h); ``bns``: k entries (weight, bias) or None; ``mode``:
    'skipsum' | 'skipconcat'; ``act``: one activation spec (see ``activation``) for all, or a list of k (PReLU: each
    module has its own weight) — entry j for layer j < k - 1, entry k - 1 for the block's activation after the skip;
    ``gates``: None or k gates (None entries allowed), indexed the same way; ``tap``: a list the k pre-activations are
    appended to."""
    k = len(convs)
    gates = gates if gates is not None else [None] * k
    acts = act if isinstance(act, list) else [act] * k
    h = x
    for j in range(k):
        h = batch_norm(convs[j](h), bns[j], eps)
        if j < k - 1:
            if tap is not None:
                tap.append(h.detach())
            h = activation(h, acts[j], gates[j])
    if mode == 'skipsum':
        h = x + h
    elif mode == 'skipconcat':
        h = torch.cat([x, h], 1)
    else:
        raise ValueError('stage_type {!r}'.format(mode))
    if tap is not None:
        tap.append(h.detach())
    return activation(h, acts[k - 1], gates[k - 1])


def skip_stage(x, blocks, mode, act, l2norm=True, gates=None, tap=None, eps=1e-5):
    """GNNSkipStage: ``blocks`` = list of (convs, bns) per block (see ``skip_block``); ``act``: one spec, or one entry
    per block (a spec or a list, see ``skip_block``); ``gates``: None or one list per block; then the row L2
    normalisation if ``l2norm``."""
    h = x
    for i, (convs, bns) in enumerate(blocks):
        a = act[i] if isinstance(act, list) else act
        h = skip_block(h, convs, bns, mode, a, gates[i] if gates is not None else None, tap, eps)
    return F.normalize(h, p=2, dim=-1) if l2norm else h
