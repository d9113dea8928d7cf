"""CPU restatement of the receding-horizon shift of mpc_warm_start_shift (include/mpc_b200.h), on arrays in the C
layouts: x, zl, zu [8N-2][B] (rows as the reference's solution.x, MPC.cpp:189-196), lambda [6N][B].  Stages 1..N-1 of
every block move to 0..N-2; the new last stage of the six state blocks of x continues with the increment of the old
last stage; actuations and multipliers repeat their last stage.  Only additions: the device gives the same bits."""
import numpy as np


def _blocks(N):
    """(first row, stages) of the eight blocks of the 8N-2 layout: x, y, psi, v, cte, epsi, delta, a."""
    return [(k * N, N) for k in range(6)] + [(6 * N, N - 1), (7 * N - 1, N - 1)]


def _shift(a, blocks, extrapolate):
    out = np.empty_like(a)
    for k, (r0, n) in enumerate(blocks):
        out[r0:r0 + n - 1] = a[r0 + 1:r0 + n]
        last = a[r0 + n - 1]
        out[r0 + n - 1] = last + (last - a[r0 + n - 2]) if extrapolate(k) else last
    return out


def shift(N, x, lam=None, zl=None, zu=None):
    """-> (x0, lam0, zl0, zu0); a multiplier array given as None comes back as None."""
    x0 = _shift(x, _blocks(N), lambda k: k < 6)
    lam0 = None if lam is None else _shift(lam, [(k * N, N) for k in range(6)], lambda k: False)
    z = [None if a is None else _shift(a, _blocks(N), lambda k: False) for a in (zl, zu)]
    return x0, lam0, z[0], z[1]
