"""fp64 numpy oracle of the kaiser-windowed sinc resampler (torchaudio.functional.resample, "kaiser_window"), given
its fp32 filter table: what the fp32 operator computes, without its rounding."""
from __future__ import annotations

import numpy as np


def resample_fp64(x, table, o: int, n: int, width: int, n_out=None):
    """(y, mag) for one signal x [L] (any float dtype, taken as fp64) and an fp32 table [n, K]:
    y[f n + p] = sum_k table[p, k] x[f o + k - width] in fp64, x = 0 outside [0, L), for the first n_out outputs
    (default ceil(n L / o); at most the (L // o + 1) n the frames give); mag = sum_k |table[p, k] x[...]|, the scale of
    an fp32 summation's error."""
    x = np.asarray(x, dtype=np.float64).reshape(-1)
    t = np.asarray(table, dtype=np.float64)
    K = t.shape[1]
    L = x.shape[0]
    xp = np.pad(x, (width, width + o))
    F = L // o + 1
    win = np.lib.stride_tricks.as_strided(xp, (F, K), (o * xp.strides[0], xp.strides[0]), writeable=False)
    n_out = -(-n * L // o) if n_out is None else n_out
    assert n_out <= F * n
    y = (win @ t.T).reshape(-1)[:n_out]
    mag = (np.abs(win) @ np.abs(t).T).reshape(-1)[:n_out]
    return y, mag
