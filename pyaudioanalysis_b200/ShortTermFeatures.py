"""Drop-in for ``pyAudioAnalysis.ShortTermFeatures`` (the three functions on the hot path).

Signatures, return types, feature names, frame-count rules and error behaviour follow the
reference (ShortTermFeatures.py:324, :389, :543); the arithmetic runs in libb200aa.so on the GPU
through the C ABI's host-buffer entry points (NumPy in, NumPy float64 out).
"""
import ctypes

import numpy as np

from . import _lib
from ._lib import lib, check, get_plan, DTYPE_I16, DTYPE_F32

PRINT_SPECTROGRAM_SHAPE = True   # the reference prints specgram.shape (ShortTermFeatures.py:451)

_CHROMA_NAMES = ['A', 'A#', 'B', 'C', 'C#', 'D', 'D#', 'E', 'F', 'F#', 'G', 'G#']


def feature_names(deltas=True):
    """The reference's feature_names list (ShortTermFeatures.py:590-604)."""
    names = ["zcr", "energy", "energy_entropy"]
    names += ["spectral_centroid", "spectral_spread"]
    names.append("spectral_entropy")
    names.append("spectral_flux")
    names.append("spectral_rolloff")
    names += ["mfcc_{0:d}".format(i) for i in range(1, 14)]
    names += ["chroma_{0:d}".format(i) for i in range(1, 13)]
    names.append("chroma_std")
    if deltas:
        names = names + ["delta " + n for n in names]
    return names


def _as_clip(signal):
    """1-D host array in one of the two device sample formats.

    int16 stays int16 (exact).  Everything else becomes float32.  The reference divides by 2**15
    and then by max |x/2**15 - mean| + 1e-10, so the features do not depend on the input scale
    as long as the clip's largest excursion from its mean is far above 2**15 * 1e-10 (about
    3.3e-6; at 1e-6 the energy row drops by an order of magnitude).  Quieter float clips keep
    the reference's scale dependence, and the GPU path reproduces it.
    """
    x = np.asarray(signal)
    if x.ndim != 1:
        x = x.reshape(-1) if x.ndim == 2 and 1 in x.shape else x
        if x.ndim != 1:
            raise ValueError("signal must be one-dimensional (mono); see audioBasicIO.stereo_to_mono")
    if x.dtype == np.int16:
        return np.ascontiguousarray(x), DTYPE_I16
    if x.dtype.kind in "iu" and x.dtype.itemsize <= 2 and (x.dtype.kind == "i" or x.dtype.itemsize == 1):
        return np.ascontiguousarray(x.astype(np.int16)), DTYPE_I16
    return np.ascontiguousarray(x.astype(np.float32)), DTYPE_F32


def _fs_int(sampling_rate):
    fs = int(sampling_rate)
    if fs != sampling_rate:
        raise ValueError("non-integer sampling rates are not supported")
    return fs


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _raise_no_frames(fs, window):
    """A clip shorter than one window: the reference has already built the mel bank (IndexError when it cannot,
    ShortTermFeatures.py:578 / :230-231) when np.concatenate finds no frames (ValueError, :684)."""
    _lib.host_table(fs, window, "mel")
    check(_lib.ERR_TOO_SHORT)


def feature_extraction(signal, sampling_rate, window, step, deltas=True):
    """Short-term features, reference ShortTermFeatures.py:543-685.

    Returns (features float64 [68|34 x n_frames], feature_names).  ``window`` / ``step`` are in
    samples and truncated with int() like the reference (:563-564).  A clip shorter than one
    window raises ValueError("need at least one array to concatenate") like :684.
    """
    window, step = int(window), int(step)
    x, code = _as_clip(signal)
    plan = get_plan(_fs_int(sampling_rate), window, step)
    T = lib().b200aa_num_frames(x.shape[0], window, step)
    if T <= 0:
        _raise_no_frames(plan.fs, window)
    F = 68 if deltas else 34
    out = np.empty((F, T), dtype=np.float32)
    check(lib().b200aa_st_features_host(plan.handle, _ptr(x), code, 1, x.shape[0], 1 if deltas else 0, _ptr(out)))
    return out.astype(np.float64), feature_names(deltas)


def spectrogram(signal, sampling_rate, window, step, plot=False, show_progress=False):
    """Reference ShortTermFeatures.py:389-452: (specgram [rows x window//2], time_axis, freq_axis)."""
    window, step = int(window), int(step)
    x, code = _as_clip(signal)
    fs = sampling_rate
    plan = get_plan(_fs_int(sampling_rate), window, step)
    K = int(window / 2)
    R = lib().b200aa_spectrogram_rows(x.shape[0], window, step)
    if R <= 0:
        check(_lib.ERR_TOO_SHORT)
    out = np.empty((R, K), dtype=np.float32)
    check(lib().b200aa_spectrogram_host(plan.handle, _ptr(x), code, x.shape[0], _ptr(out)))
    specgram = out.astype(np.float64)
    freq_axis = [float((f + 1) * fs) / (2 * K) for f in range(K)]
    time_axis = [float(t * step) / fs for t in range(R)]
    if plot:
        _plot(specgram.transpose()[::-1, :])
    if PRINT_SPECTROGRAM_SHAPE:
        print(specgram.shape)
    return specgram, time_axis, freq_axis


def chromagram(signal, sampling_rate, window, step, plot=False, show_progress=False):
    """Reference ShortTermFeatures.py:324-386: (chromogram [rows x 12], time_axis, chroma names)."""
    window, step = int(window), int(step)
    x, code = _as_clip(signal)
    fs = sampling_rate
    plan = get_plan(_fs_int(sampling_rate), window, step)
    R = lib().b200aa_chromagram_rows(x.shape[0], window, step)
    if R <= 0 or x.shape[0] - step - window < 0:
        check(_lib.ERR_TOO_SHORT)
    out = np.empty((R, 12), dtype=np.float32)
    check(lib().b200aa_chromagram_host(plan.handle, _ptr(x), code, x.shape[0], _ptr(out)))
    chromogram = out.astype(np.float64)
    time_axis = [(t * step) / fs for t in range(R)]
    if plot:
        _plot(chromogram.transpose()[::-1, :])
    return chromogram, time_axis, list(_CHROMA_NAMES)


def _plot(image):
    try:
        import matplotlib.pyplot as plt
    except ImportError as exc:   # the reference needs matplotlib for plot=True as well
        raise ImportError("plot=True needs matplotlib") from exc
    plt.imshow(image)
    plt.colorbar()
    plt.show()
