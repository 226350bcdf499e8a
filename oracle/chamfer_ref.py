"""ORACLE (test infrastructure, NOT product code) -- Chamfer distance on the CPU, float64, brute force.

The reference has no Chamfer loss (run.py:629-630 only names it as an option); this restates the textbook definition the product
kernel (geniconet_b200/csrc/gin_chamfer.cuh) implements, in difference form over every pair:

    d_xy[b,i] = min_j |x[b,i] - y[b,j]|^2,  idx_xy[b,i] = the lowest j reaching it;  d_yx / idx_yx the same from y towards x
    dx_i = 2 g_xy_i (x_i - y_idx_xy(i)) + sum_{j : idx_yx(j) = i} 2 g_yx_j (x_i - y_j),  dy symmetrically.
"""
import numpy as np


def _nn(a, b, chunk):
    """a [N,3], b [M,3] float64 -> (min squared distance [N], argmin [N] int64, lowest index on ties)."""
    d = np.empty(a.shape[0])
    idx = np.empty(a.shape[0], dtype=np.int64)
    for s in range(0, a.shape[0], chunk):
        diff = a[s:s + chunk, None, :] - b[None, :, :]
        sq = (diff * diff).sum(-1)
        idx[s:s + chunk] = sq.argmin(1)
        d[s:s + chunk] = sq.min(1)
    return d, idx


def nearest(x, y, chunk=512):
    """x [B,N,3], y [B,M,3] -> (d_xy [B,N] float64, idx_xy [B,N] int64): one direction."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    d, i = zip(*(_nn(x[b], y[b], chunk) for b in range(x.shape[0])))
    return np.stack(d), np.stack(i)


def chamfer_forward(x, y, chunk=512):
    """x [B,N,3], y [B,M,3] -> (d_xy [B,N], idx_xy [B,N], d_yx [B,M], idx_yx [B,M]) in float64 / int64."""
    return nearest(x, y, chunk) + nearest(y, x, chunk)


def pair_distance(x, y, idx):
    """Squared float64 distance of x[b,i] to y[b, idx[b,i]]."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    yy = np.take_along_axis(y, np.asarray(idx, dtype=np.int64)[..., None].repeat(3, -1), axis=1)
    return ((x - yy) ** 2).sum(-1)


def chamfer_backward(x, y, idx_xy, idx_yx, g_xy=None, g_yx=None):
    """Gradients (dx [B,N,3], dy [B,M,3]) of sum(g_xy * d_xy) + sum(g_yx * d_yx) for the given nearest-neighbour indices."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    dx, dy = np.zeros_like(x), np.zeros_like(y)
    for b in range(x.shape[0]):
        if g_xy is not None:
            j = np.asarray(idx_xy[b], dtype=np.int64)
            t = 2.0 * np.asarray(g_xy[b], dtype=np.float64)[:, None] * (x[b] - y[b][j])
            dx[b] += t
            np.add.at(dy[b], j, -t)
        if g_yx is not None:
            i = np.asarray(idx_yx[b], dtype=np.int64)
            t = 2.0 * np.asarray(g_yx[b], dtype=np.float64)[:, None] * (y[b] - x[b][i])
            dy[b] += t
            np.add.at(dx[b], i, -t)
    return dx, dy
