"""Reference of the persistence spectrum (integer data): a per-column bincount in numpy.

Definition (include/spx.h, spx_stft_exec_persistence): for uint8 waterfall rows [S*F][N] (stream s owns rows
s*F .. s*F+F-1; the levels are SURVEY A7's index, ``oracle.spectral_ref.waterfall_u8``)

    counts[s][q][j] = #{f in [0, F) : rows[s*F + f][j] == q}        uint32 [S][256][N]

so level q covers dB values in [vmin + q*D, vmin + (q+1)*D) with D = (vmax - vmin)/256, level 0 also holds values
below vmin and NaN, level 255 values at or above vmax - D, and every column sums to F."""
import numpy as np


def persistence(q_rows, n_streams: int = 1) -> np.ndarray:
    q = np.asarray(q_rows, dtype=np.uint8)
    n = q.shape[-1]
    q = q.reshape(n_streams, -1, n)
    out = np.zeros((n_streams, 256, n), np.uint32)
    cols = np.arange(n)
    for s in range(n_streams):
        flat = (q[s].astype(np.int64) * n + cols).reshape(-1)   # one bincount over (level, column) pairs
        out[s] = np.bincount(flat, minlength=256 * n).reshape(256, n)
    return out
