"""The handful of ``cfg`` keys the hot-path layers read at construction time
(ref: graphgym/config.py:316-372,409-420; read sites idconv.py:19,25 and layer.py:23-34).

yacs is not a dependency of this package; ``cfg`` is a plain attribute tree with the reference's
defaults, and ``load_cfg(path)`` merges one of the reference's ``config/*_tf/*.yaml`` files.
"""
import yaml


class _Node(dict):
    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    def __setattr__(self, k, v):
        self[k] = v


def _defaults():
    c = _Node()
    c.gnn = _Node(layers_pre_mp=0, layers_mp=2, layers_post_mp=0, dim_inner=16, layer_type='generalconv',
                  stage_type='stack', batchnorm=True, act='relu', dropout=0.0, agg='add',
                  normalize_adj=False, l2norm=True, keep_edge=0.5, self_msg='concat', att_heads=1,
                  skip_every=1, msg_direction='single')
    c.bn = _Node(eps=1e-5, mom=0.1)
    c.mem = _Node(inplace=False)
    c.dataset = _Node(transform='none', augment_feature=[], augment_feature_dims=[], edge_dim=128)
    c.train = _Node(batch_size=16)
    c.num_threads = 6
    c.device = 'auto'
    # not a reference key: storage type of the operand the aggregation gathers.  'f32' = the reference's arithmetic
    # (1e-5 parity); 'bf16' = the north star's 1e-2 mode (rows gathered in bf16, fp32 products and sums)
    # fused_postops: GeneralLayer's BN / activation / L2 as one fused pass (False = the nn modules one by one)
    c.b200 = _Node(gather_dtype='f32', fused_postops=True)
    return c


cfg = _defaults()


def reset_cfg():
    cfg.clear()
    cfg.update(_defaults())


def _merge(dst, src):
    for k, v in src.items():
        if isinstance(v, dict):
            node = dst.get(k)
            if not isinstance(node, _Node):
                node = _Node()
                dst[k] = node
            _merge(node, v)
        else:
            dst[k] = v


def load_cfg(path):
    """Merge a reference yaml (e.g. config/gcnconv_tf/*.yaml) into ``cfg``."""
    with open(path) as f:
        data = yaml.safe_load(f) or {}
    _merge(cfg, data)
    return cfg
