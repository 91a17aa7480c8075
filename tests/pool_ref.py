"""Reference of the pooled spectrogram (display detectors), float64 numpy.

Definition (include/spx.h, spx_stft_exec_pooled / spx_pool_finalize): for stream s, frame f (0 <= f < F) and bin j
(fftshift order) let P[f][j] = |X_f[j]|^2.  With K >= 1 frames per row and B >= 1 bins per column (N % B == 0),
C = N / B and G = ceil(F / K); row g pools the frames [gK, min((g+1)K, F)) (the last row may hold fewer) and column c
the bins [cB, (c+1)B).

  mean: the mean of P over the cell's n_g * B values (NaN propagates, as in welch_acc)
  max:  the maximum of P over the cell (NaN skipped, as in maxhold; a cell of nothing but NaN is -inf dB)
  dB = 20 log10(sqrt(P) + eps)                      (the row definition, so K = B = 1 gives back the dB rows)
  level = oracle.spectral_ref.waterfall_u8(dB as float32, vmin, vmax)

Two forms: ``pool_power`` / ``pool_db`` apply it to power rows (the float64 oracle), ``pool_db_rows`` to float32 dB
rows, recovering the power as (10^(d/20) - eps)^2 clipped at 0 (the rows of the same call)."""
import numpy as np

EPS = np.float64(np.float32(1e-12))   # the plans' db_eps (float32) as the library uses it


def _cells(a, K, B, n_streams):
    """[S][G] lists of the float64 cell blocks [n_g, C, B] of rows [S*F, N]."""
    a = np.asarray(a, np.float64)
    N = a.shape[-1]
    a = a.reshape(n_streams, -1, N)
    F = a.shape[1]
    G = -(-F // K)
    return a, F, G, N // B


def pool_power(P, K, B, mode, n_streams=1):
    """Pooled power [S, G, C] of power rows [S*F, N]; a max cell of nothing but NaN is NaN here (-inf dB in pool_db)."""
    a, F, G, C = _cells(P, K, B, n_streams)
    out = np.empty((n_streams, G, C))
    for g in range(G):
        cell = a[:, g * K:min((g + 1) * K, F)].reshape(n_streams, -1, C, B)
        if mode == "mean":
            out[:, g] = cell.mean(axis=(1, 3))
        else:
            out[:, g] = np.fmax.reduce(np.fmax.reduce(cell, axis=3), axis=1)
    return out


def _power_to_db(p, eps):
    with np.errstate(divide="ignore", invalid="ignore"):
        return 20 * np.log10(np.sqrt(p) + eps)


def pool_db(P, K, B, mode, n_streams=1, eps=EPS):
    """Pooled dB [S, G, C] of power rows."""
    p = pool_power(P, K, B, mode, n_streams)
    d = _power_to_db(p, eps)
    if mode == "max":
        d = np.where(np.isnan(p), -np.inf, d)
    return d


def db_to_power(d, eps=EPS):
    """The power a dB row value encodes: (10^(d/20) - eps)^2, clipped at 0 (NaN stays NaN)."""
    d = np.asarray(d, np.float64)
    a = 10 ** (d / 20) - eps
    return np.where(a < 0, 0.0, a) ** 2


def pool_db_rows(db_rows, K, B, mode, n_streams=1, eps=EPS):
    """Pooled dB [S, G, C] of float32 dB rows [S*F, N].  max: the largest dB value of the cell itself (dB is monotonic
    in power), so it equals the rows' own maximum bit for bit."""
    if mode == "max":
        a, F, G, C = _cells(db_rows, K, B, n_streams)
        out = np.empty((n_streams, G, C))
        for g in range(G):
            cell = a[:, g * K:min((g + 1) * K, F)].reshape(n_streams, -1, C, B)
            out[:, g] = np.fmax.reduce(np.fmax.reduce(cell, axis=3), axis=1)
        return np.where(np.isnan(out), -np.inf, out)
    return pool_db(db_to_power(db_rows, eps), K, B, "mean", n_streams, eps)
