"""CPU restatement of ID-GNN Fast's cycle features (TEST INFRASTRUCTURE ONLY).

``compute_identity`` follows graphgym/contrib/transform/identity.py:25-35: A_hat = D^-1/2 (A+I) D^-1/2
(``norm`` at :7-22, remaining self loops, degree over edge_index[0]), densified, and
diag(A_hat^p) for p = 1..k by repeated dense matmul.  ``closed_walks`` is the integer variant the
north star names (diag(A^p), exact int64) — the reference itself never computes it (SURVEY D2).
``diag_powers_sparse`` is the same A_hat's diagonal powers for chosen source nodes without densifying, for graphs far
past the dense form's reach (on the device of the edge list).
"""
import numpy as np
import torch

from .layers import gcn_norm_src


def compute_identity(edge_index, n, k, dtype=torch.float32):
    ei, value = gcn_norm_src(edge_index, n, dtype)
    adj = torch.zeros((n, n), dtype=dtype)
    adj.index_put_((ei[0], ei[1]), value, accumulate=True)  # sparse -> dense sums duplicates
    diag_all = [torch.diag(adj)]
    power = adj
    for _ in range(1, k):
        power = power @ adj
        diag_all.append(torch.diag(power))
    return torch.stack(diag_all, dim=1)


def diag_powers_sparse(edge_index, n, k, sources, chunk=1 << 21):
    """[len(sources), k] float64: diag(A_hat^p)[sources] for p = 1..k with the A_hat of ``compute_identity``, by k hops
    V <- A_hat V from the sources' unit columns (gather / scale / index_add_ over edge chunks)."""
    ei, value = gcn_norm_src(edge_index, n, torch.float64)
    row, col = ei
    dev = edge_index.device
    s = torch.as_tensor(sources, device=dev).long()
    cols = torch.arange(s.numel(), device=dev)
    v = torch.zeros((n, s.numel()), dtype=torch.float64, device=dev)
    v[s, cols] = 1.0
    out = torch.empty((s.numel(), k), dtype=torch.float64, device=dev)
    for p in range(k):
        nxt = torch.zeros_like(v)
        for a in range(0, row.numel(), chunk):
            b = min(row.numel(), a + chunk)
            nxt.index_add_(0, row[a:b], v.index_select(0, col[a:b]) * value[a:b].view(-1, 1))
        v = nxt
        out[:, p] = v[s, cols]
    return out


def closed_walks(edge_index, n, k):
    """diag(A^p), p = 1..k, exact int64; A[src, tgt] counts duplicate edges (multigraph)."""
    ei = np.asarray(edge_index, dtype=np.int64)
    a = np.zeros((n, n), dtype=np.int64)
    np.add.at(a, (ei[0], ei[1]), 1)
    out = np.zeros((n, k), dtype=np.int64)
    p = np.eye(n, dtype=np.int64)
    for i in range(k):
        p = p @ a
        out[:, i] = np.diag(p)
    return out
