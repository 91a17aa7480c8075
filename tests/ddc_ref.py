"""float64 numpy statement of the DDC definition (include/spx.h, spx_ddc_*): the oracle of the DDC tests.

  phi(n) = ((first_sample + n) * phase_inc) mod 2^64         numpy uint64 wrapping multiplication
  mix[n] = x[n] * exp(-2 pi i phi(n) / 2^64)
  y      = np.convolve(mix, h, 'valid')[::D]                 float64 taps, as the STFT oracle uses the float64 window
"""
import numpy as np


def phases(n_samples, first_sample, phase_inc):
    """phi(n) of n = 0 .. n_samples - 1 as uint64 (exact, wrapping)."""
    n = np.arange(n_samples, dtype=np.uint64) + np.uint64(first_sample)
    with np.errstate(over="ignore"):
        return n * np.uint64(int(phase_inc) % (1 << 64))


def nco(n_samples, first_sample, phase_inc):
    """exp(-2 pi i phi(n) / 2^64), complex128."""
    return np.exp(-2j * np.pi * (phases(n_samples, first_sample, phase_inc).astype(np.float64) / 2.0 ** 64))


def to_complex(x, in_scale=1.0):
    """complex128 samples of complex input or interleaved int16 I, Q, times in_scale."""
    x = np.asarray(x)
    if x.dtype == np.int16:
        x = x.astype(np.float64).reshape(-1, 2)
        x = x[:, 0] + 1j * x[:, 1]
    return x.astype(np.complex128) * in_scale


def ddc(x, taps, decim, phase_inc, first_sample=0, in_scale=1.0):
    """y[m] of the definition, complex128 [M]."""
    xc = to_complex(x, in_scale)
    h = np.asarray(taps, np.float64)
    if xc.size < h.size:
        return np.zeros(0, np.complex128)
    mix = xc * nco(xc.size, first_sample, phase_inc)
    return np.convolve(mix, h, "valid")[::int(decim)]


def bound(taps, x, in_scale=1.0):
    """sum |h| * max |x|: the scale of the parity bar (1e-5 of it)."""
    xc = to_complex(x, in_scale)
    return float(np.abs(np.asarray(taps, np.float64)).sum() * (np.abs(xc).max() if xc.size else 0.0))
