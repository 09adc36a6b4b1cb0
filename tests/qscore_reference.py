"""numpy restatement of what ddz_q_features computes (TEST INFRASTRUCTURE): the first-layer features of the reference's
NetComplicated family (net.py:65-139) from per-rank nibbles and the lookup tables of agent.q_tables, without ever building
the [n, C+1, 15, 4] input.  tests/ checks it against the torch module's float64 convolutions on the CPU, for left-aligned
rows and for form-B rows (test_consumer_contract.py, test_q_features_kernel.py), so the table construction and the formulas
are validated where there is no GPU.  The CUDA kernel is checked against the torch module directly, on the GPU
(test_q_features_kernel.py)."""
import numpy as np

LUT = np.zeros((16, 4))
for _c in range(5):
    LUT[_c, :_c] = 1.0
    LUT[8 + _c, 4 - _c:] = 1.0


def features(nibbles, scales, T, rank_bias, L, line_bias):
    """nibbles int [n, C+1, 15], scales float [n, C+1] (1 except the two probability planes) -> float64 [n, 19 W]:
    [W x 15 rank features (o * 15 + r) | W x 4 line features (o * 4 + j)], the layout of net.py:93-97's x"""
    T, rank_bias, L, line_bias = (np.asarray(a, np.float64) for a in (T, rank_bias, L, line_bias))
    n, cin, _ = nibbles.shape
    W = T.shape[2]                                                                # T [C+1, 16, W, 4], rank_bias [W, 4]
    rank = np.broadcast_to(rank_bias[None, None], (n, 15, W, 4)).copy()          # [n, r, o, k]
    line = np.broadcast_to(line_bias[None, :, None], (n, W, 4)).copy()           # [n, o, j]
    for c in range(cin):
        t = T[c][nibbles[:, c, :]]                                                # [n, 15, W, 4]
        rank += scales[:, c, None, None, None] * t
        lw = L[c][None] * scales[:, c, None, None]                                # [n, 15, W]
        line += np.einsum("nro,nrj->noj", lw, LUT[nibbles[:, c, :]])
    pooled = rank.max(axis=3)                                                     # MaxPool2d((1, 4)) over the four convs
    return np.concatenate([pooled.transpose(0, 2, 1).reshape(n, -1), line.reshape(n, -1)], axis=1)


def nibbles_of(x):
    """float [n, C+1, 15, 4] thermometer rows (possibly scaled) -> (nibbles int [n, C+1, 15], scales [n, C+1]); a row whose
    ones are right-aligned (form B's probability planes: slot 0 empty, slot 3 set) gets 8 + count, its entry of LUT"""
    x = np.asarray(x, np.float64)
    nib = (x > 0).sum(-1)
    nib = np.where((x[..., 0] == 0) & (x[..., 3] > 0), 8 + nib, nib)
    scale = x.max(axis=(-1, -2))
    scale[scale == 0] = 1.0
    return nib, scale
