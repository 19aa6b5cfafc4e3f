"""Shared test helpers: seeded graphs and the parity metric."""
import numpy as np
import torch


def random_graph(seed, n, e, loops=0, dups=0, symmetric=False):
    g = torch.Generator().manual_seed(seed)
    src = torch.randint(0, n, (e,), generator=g)
    tgt = torch.randint(0, n, (e,), generator=g)
    if loops:
        lp = torch.randint(0, n, (loops,), generator=g)
        src, tgt = torch.cat([src, lp]), torch.cat([tgt, lp])
    if dups:
        src, tgt = torch.cat([src, src[:dups]]), torch.cat([tgt, tgt[:dups]])
    if symmetric:
        src, tgt = torch.cat([src, tgt]), torch.cat([tgt, src])
    perm = torch.randperm(src.numel(), generator=g)
    return torch.stack([src[perm], tgt[perm]])


def powerlaw_graph(seed, n, avg_deg, max_deg=None, exponent=2.1):
    """Chung-Lu style symmetric graph with a power-law expected degree sequence (hub rows)."""
    rng = np.random.default_rng(seed)
    w = (np.arange(1, n + 1, dtype=np.float64)) ** (-1.0 / (exponent - 1.0))
    w *= avg_deg * n / w.sum()
    if max_deg:
        w = np.minimum(w, max_deg)
    p = w / w.sum()
    m = int(avg_deg * n / 2)
    a = rng.choice(n, size=m, p=p)
    b = rng.choice(n, size=m, p=p)
    perm = rng.permutation(n)  # hubs are not the low ids
    a, b = perm[a], perm[b]
    ei = np.stack([np.concatenate([a, b]), np.concatenate([b, a])])
    return torch.from_numpy(ei.astype(np.int64))


def rel_err(a, b):
    """max |a-b| / max(|b|, tiny): the norm-wise relative error used for every fp parity check.  Not enough alone where the
    rows or columns differ in scale (hub rows of a sum aggregation, high powers of compute_identity): the largest one sets
    the denominator and hides errors in the small ones; bound each element by its own scale there as well."""
    a = torch.as_tensor(a, dtype=torch.float64).cpu()
    b = torch.as_tensor(b, dtype=torch.float64).cpu()
    assert a.shape == b.shape, (a.shape, b.shape)
    if b.numel() == 0:
        return 0.0
    return float((a - b).abs().max() / b.abs().max().clamp(min=1e-30))


FP32_TOL = 1e-5  # north_star: "within 1e-5 relative (fp32)"
