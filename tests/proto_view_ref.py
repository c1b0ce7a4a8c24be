"""float64 reference of the exact-mode prototype sums over a global view (bacs_proto_accumulate_view).

The reference's ``features[mask.expand(..)].view(D, -1).sum(-1)`` places element k of the run of image b, channel c
and task t at flat position D * (pre + pre_bt) + c * n_bt + k of a D x N view and adds it to row position // N.  One
process has pre = 0 and N = N_t; a data-parallel rank sees its images through pre = view_pre[t] (the pixels of task t
in the images of the ranks below it) and N = view_n[t] (the pixels over all ranks)."""
import numpy as np
import torch


def exact_view_sums(feat, task, T, view=None):
    """feat [B,D,h,w] (any float dtype), task [B,h,w] (int, -1 = no task), view = (view_pre, view_n) int arrays of T
    entries or None (the local view).  Returns (sums fp64 [T,D], |addend| sums fp64 [T,D], counts int64 [T])."""
    x = torch.as_tensor(feat).detach().cpu().double()
    B, D = x.shape[:2]
    xf = x.reshape(B, D, -1)
    tf = torch.as_tensor(np.asarray(task)).reshape(B, -1)
    S = torch.zeros(T, D, dtype=torch.float64)
    A = torch.zeros(T, D, dtype=torch.float64)
    counts = torch.zeros(T, dtype=torch.int64)
    for t in range(T):
        m = tf == t
        n_b = m.sum(1)
        counts[t] = int(n_b.sum())
        if counts[t] == 0:
            continue
        pre, N = (0, int(counts[t])) if view is None else (int(view[0][t]), int(view[1][t]))
        for b in range(B):
            nb = int(n_b[b])
            if nb:
                vals = xf[b][:, m[b]]                                               # [D, nb], pixel order
                pos = D * pre + torch.arange(D).unsqueeze(1) * nb + torch.arange(nb).unsqueeze(0)
                rows = (pos // N).reshape(-1)
                S[t].index_add_(0, rows, vals.reshape(-1))
                A[t].index_add_(0, rows, vals.abs().reshape(-1))
            pre += nb
    return S, A, counts


def shard_views(n_bt, bounds):
    """Global view of every shard [bounds[i], bounds[i+1]) of a batch whose per-image task counts are n_bt [B,T]."""
    n = np.asarray(n_bt, dtype=np.int64)
    tot = n.sum(0)
    return [(n[:lo].sum(0), tot.copy()) for lo in bounds[:-1]]
