"""float64 numpy statement of the channelizer definition (include/spx.h, spx_chan_*): the oracle of the channelizer tests.

Channel j (fftshift order, c = j - M/2) is the DDC of tests/ddc_ref.py with phase_inc_j = c 2^64 / M, taps h and
decimation D.  Written twice: ``channelize`` as the polyphase fold by global sample class plus ``np.fft.fft`` read out in
fftshift order, and ``channelize_ddc`` as M runs of ``ddc_ref.ddc``.
"""
import numpy as np

from tests import ddc_ref


def out_count(n_samples, T, D):
    return 0 if n_samples < T else (n_samples - T) // D + 1


def phase_inc(j, M):
    """phase_inc_j = (j - M/2) 2^64 / M as a two's-complement int64."""
    v = ((j - M // 2) * ((1 << 64) // M)) % (1 << 64)
    return v - (1 << 64) if v >= 1 << 63 else v


def channelize(x, taps, M, D, first_sample=0, in_scale=1.0):
    """y[j][m], complex128 [M][n_out]: fold v_m[r] = sum of h[k] x[mD + T-1-k] over the taps whose sample has global class
    r = (first_sample + mD + T-1-k) mod M, then the M-point DFT of v_m in fftshift order."""
    xc = ddc_ref.to_complex(x, in_scale)
    h = np.asarray(taps, np.float64)
    T = h.size
    n_out = out_count(xc.size, T, D)
    if n_out == 0:
        return np.zeros((M, 0), np.complex128)
    g = h[::-1]                                           # g[j] = h[T-1-j]: window offset j holds sample mD + j
    idx = np.arange(n_out)[:, None] * D + np.arange(T)[None, :]
    prod = xc[idx] * g[None, :]                           # [n_out][T]
    cls = (first_sample % M + idx) % M                    # global class of each sample
    v = np.zeros((n_out, M), np.complex128)
    rows = np.broadcast_to(np.arange(n_out)[:, None], idx.shape)
    np.add.at(v, (rows, cls), prod)
    return np.fft.fftshift(np.fft.fft(v, axis=1), axes=1).T.copy()


def channelize_ddc(x, taps, M, D, first_sample=0, in_scale=1.0, channels=None):
    """The same as M (or ``channels``) DDCs of ddc_ref, complex128 [len(channels)][n_out]."""
    js = range(M) if channels is None else channels
    return np.stack([ddc_ref.ddc(x, taps, D, phase_inc(j, M), first_sample, in_scale) for j in js])


def bound(taps, x, in_scale=1.0):
    """sum |h| max |x|: the scale of the parity bar (1e-5 of it), as for the DDC."""
    return ddc_ref.bound(taps, x, in_scale)
