"""NumPy float64 restatement of pyAudioAnalysis' short-term / mid-term feature path.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``): this is the checker the
CUDA path is compared against and the CPU baseline ``bench.py`` times.  It is
never on the product path.

Parity status: PINNED.  ``tests/test_oracle_golden.py`` checks every function
here against golden vectors produced by the unmodified reference
(``/root/reference`` imported through ``oracle/ref_import.py``; generator:
``oracle/make_golden.py``; fixtures: ``tests/golden/*.npz``).  The reference's
own tests pin shapes only (pytests/test_feature_extraction.py:14-15,27-28;
those shape pins are reproduced in ``tests/test_oracle_golden.py::
test_reference_pytest_inputs``).  ``tests/test_oracle_vs_reference.py`` additionally holds the oracle to
the reference's values on randomised configurations and error cases
(``tests/golden/vs_reference.npz``, generator ``oracle/make_golden_vs_reference.py``).

Third-party arithmetic: the reference takes its DFT and DCT from SciPy
(``scipy.fftpack.fft`` ShortTermFeatures.py:5,617 and
``scipy.fftpack.realtransforms.dct`` :8,253; requirements.txt only pins
``scipy>=1.6.3``).  Both are the textbook definitions (unnormalised forward DFT
``X[k] = sum_n x[n] exp(-2 pi i k n / N)``; orthonormal DCT-II).  Here the DFT
is ``numpy.fft`` (same pocketfft family) and the DCT is an explicit cosine
matrix; ``oracle/dft_def.c`` restates both definitions naively in C and
``tests/test_oracle_golden.py`` pins numpy against it.

Two flavours are provided:

* ``*_loop`` functions walk the frames one by one and redo the loop-invariant
  table work per frame exactly as often as the reference does (the reference
  recomputes its chroma tables for every frame, ShortTermFeatures.py:281-282).
  They have the reference's cost profile and are what ``bench.py`` times as the
  CPU baseline (kind="port").
* the un-suffixed functions are vectorised over frames; they are the fast
  checker for the parity tests.  Both flavours are tested against each other
  and against the golden vectors.

Every function cites the reference lines it follows (paths relative to
/root/reference/pyAudioAnalysis/).
"""
from __future__ import annotations

import math
import sys

import numpy as np

EPS = sys.float_info.epsilon  # ShortTermFeatures.py:11

N_MEL = 40          # 13 linear + 27 log filters, ShortTermFeatures.py:191-192
N_MFCC = 13         # ShortTermFeatures.py:582
N_BASE = 34         # 8 + 13 + 13, ShortTermFeatures.py:580-585
CHROMA_NAMES = ['A', 'A#', 'B', 'C', 'C#', 'D', 'D#', 'E', 'F', 'F#', 'G', 'G#']  # :283-284


# --------------------------------------------------------------------------- names
def feature_names(deltas: bool = True) -> list[str]:
    """ShortTermFeatures.py:590-604."""
    base = ["zcr", "energy", "energy_entropy", "spectral_centroid", "spectral_spread",
            "spectral_entropy", "spectral_flux", "spectral_rolloff"]
    base += [f"mfcc_{i:d}" for i in range(1, N_MFCC + 1)]
    base += [f"chroma_{i:d}" for i in range(1, 13)]
    base.append("chroma_std")
    if deltas:
        return base + ["delta " + b for b in base]
    return base


def mid_feature_names(st_names: list[str]) -> list[str]:
    """MidTermFeatures.py:113-114."""
    return [n + "_mean" for n in st_names] + [n + "_std" for n in st_names]


# --------------------------------------------------------------------------- clip normalisation
def normalize_clip(signal) -> np.ndarray:
    """ShortTermFeatures.py:567-570 + dc_normalize :14-19.

    ``/2**15`` is applied to every dtype, then the whole clip is centred on its
    mean and divided by (max |.| + 1e-10).
    """
    y = np.asarray(signal, dtype=np.float64) / 32768.0
    y = y - y.mean()
    y = y / (np.abs(y).max() + 1e-10)
    return y


def frame_count(n_samples: int, window: int, step: int) -> int:
    """Loop guard ``cur + window - 1 < N`` at ShortTermFeatures.py:608."""
    if n_samples < window:
        return 0
    return (n_samples - window) // step + 1


# --------------------------------------------------------------------------- host tables
def mel_filterbank(fs, n_bins: int) -> np.ndarray:
    """ShortTermFeatures.py:191-233 (mfcc_filter_banks) -> [40, n_bins] float64.

    The reference passes ``num_fft = window//2`` as if it were the FFT size, so
    the bin-frequency grid is ``k * fs / n_bins`` (:215) and edge indices are
    ``floor(f * n_bins / fs) + 1`` (:222-228).  Kept as is.
    """
    low, lin_step, log_ratio, n_lin, n_log = 133.33, 200 / 3, 1.0711703, 13, 27
    n_filt = n_lin + n_log
    edges = np.zeros(n_filt + 2)
    edges[:n_lin] = low + np.arange(n_lin) * lin_step
    edges[n_lin:] = edges[n_lin - 1] * log_ratio ** np.arange(1, n_log + 3)
    peak = 2.0 / (edges[2:] - edges[:-2])
    grid = np.arange(n_bins) / (1.0 * n_bins) * fs
    bank = np.zeros((n_filt, n_bins))
    for i in range(n_filt):
        lo, ce, hi = edges[i], edges[i + 1], edges[i + 2]
        k_lo = int(np.floor(lo * n_bins / fs)) + 1
        k_ce = int(np.floor(ce * n_bins / fs)) + 1
        k_hi = int(np.floor(hi * n_bins / fs)) + 1
        up = np.arange(k_lo, k_ce, dtype=int)
        down = np.arange(k_ce, k_hi, dtype=int)
        # out-of-range bins raise IndexError exactly like the reference's fancy store
        bank[i][up] = (peak[i] / (ce - lo)) * (grid[up] - lo)
        bank[i][down] = (peak[i] / (hi - ce)) * (hi - grid[down])
    return bank


def dct_matrix(n_out: int = N_MFCC, n_in: int = N_MEL) -> np.ndarray:
    """Orthonormal DCT-II rows 0..n_out-1 (scipy dct(type=2, norm='ortho'), :253)."""
    n = np.arange(n_in)
    k = np.arange(n_out)[:, None]
    mat = np.cos(np.pi * k * (2 * n + 1) / (2.0 * n_in)) * math.sqrt(2.0 / n_in)
    mat[0, :] = math.sqrt(1.0 / n_in)
    return mat


def chroma_tables(fs, n_bins: int):
    """ShortTermFeatures.py:257-274 (chroma_features_init).

    Returns (semitone index per bin, number of bins sharing that semitone).
    """
    freqs = np.array([((k + 1) * fs) / (2 * n_bins) for k in range(n_bins)])
    semis = np.round(12.0 * np.log2(freqs / 27.50)).astype(int)
    share = np.zeros((n_bins,))
    for u in np.unique(semis):
        where = np.nonzero(semis == u)
        share[where] = where[0].shape
    return semis, share


def chroma_operator(fs, n_bins: int) -> np.ndarray:
    """The fixed linear map hidden in chroma_features (:285-302) as a dense [12, n_bins] matrix.

    ``C[semis] = X**2`` is a fancy store: for duplicate targets the LAST source
    bin wins and negative targets wrap around (numpy indexing); then
    ``C /= share[semis]`` divides slot j by ``share[semis[j]]`` (sic), and the
    slots are folded modulo 12.  Raises ValueError where the reference does
    (its else-branch :290-294 cannot succeed).
    """
    semis, share = chroma_tables(fs, n_bins)
    if not semis.max() < n_bins:
        raise ValueError("chroma: semitone index >= num_fft (window too short for this "
                         "sampling rate; the reference raises here as well)")
    winner = np.full(n_bins, -1, dtype=int)
    for k in range(n_bins):               # ascending k => last store wins
        winner[semis[k]] = k              # negative semis wrap like numpy
    op = np.zeros((12, n_bins))
    for j in range(n_bins):
        if winner[j] >= 0:
            op[j % 12, winner[j]] += 1.0 / share[semis[j]]
    return op


# --------------------------------------------------------------------------- per-frame pieces (loop flavour)
def _zcr(x):
    """ShortTermFeatures.py:22-26."""
    flips = np.sum(np.abs(np.diff(np.sign(x)))) / 2
    return np.float64(flips) / np.float64(len(x) - 1.0)


def _energy(x):
    """ShortTermFeatures.py:29-31."""
    return np.sum(x ** 2) / np.float64(len(x))


def _block_entropy(v, n_blocks=10):
    """ShortTermFeatures.py:34-51 and :85-107 (same recipe on samples / on |X|)."""
    total = np.sum(v ** 2)
    blk = int(np.floor(len(v) / n_blocks))
    body = v[0:blk * n_blocks]
    parts = body.reshape(n_blocks, blk)           # row j = v[j*blk:(j+1)*blk]
    s = np.sum(parts ** 2, axis=1) / (total + EPS)
    return -np.sum(s * np.log2(s + EPS))


def _centroid_spread(X, fs):
    """ShortTermFeatures.py:57-82."""
    ind = np.arange(1, len(X) + 1) * (fs / (2.0 * len(X)))
    top = X.max()
    Xt = X / EPS if top == 0 else X / top
    den = np.sum(Xt) + EPS
    cen = np.sum(ind * Xt) / den
    spr = np.sqrt(np.sum(((ind - cen) ** 2) * Xt) / den)
    return cen / (fs / 2.0), spr / (fs / 2.0)


def _flux(X, Xp):
    """ShortTermFeatures.py:110-124."""
    return np.sum((X / np.sum(X + EPS) - Xp / np.sum(Xp + EPS)) ** 2)


def _rolloff(X, c=0.90):
    """ShortTermFeatures.py:127-140."""
    e = np.sum(X ** 2)
    over = np.nonzero(np.cumsum(X ** 2) + EPS > c * e)[0]
    return np.float64(over[0]) / float(len(X)) if len(over) > 0 else 0.0


def _chroma_frame(X, fs, n_bins, tabs=None):
    """ShortTermFeatures.py:277-321 with the scatter written out as the reference does it."""
    semis, share = chroma_tables(fs, n_bins) if tabs is None else tabs
    spec = X ** 2
    if not semis.max() < semis.shape[0]:
        raise ValueError("chroma: semitone index >= num_fft")
    C = np.zeros((semis.shape[0],))
    C[semis] = spec
    C /= share[semis]
    padded = np.zeros((int(np.ceil(C.shape[0] / 12.0) * 12),))
    padded[0:C.shape[0]] = C
    out = padded.reshape(-1, 12).sum(axis=0)
    tot = spec.sum()
    return out / (EPS if tot == 0 else tot)


def _spectrum(frame, n_bins):
    """ShortTermFeatures.py:617-621: |FFT|[0:K] / K (full complex transform, like the reference)."""
    return np.abs(np.fft.fft(frame))[0:n_bins] / n_bins


def feature_extraction_loop(signal, fs, window, step, deltas=True, tables_per_frame=True):
    """Frame-by-frame restatement of ShortTermFeatures.py:543-685.

    ``tables_per_frame=True`` redoes the chroma tables for every frame, which
    is what the reference does (:281-282) and what dominates its run time.
    """
    window, step = int(window), int(step)
    y = normalize_clip(signal)
    n = len(y)
    K = int(window / 2)
    bank = mel_filterbank(fs, K)
    dmat = dct_matrix()
    fixed_tabs = None if tables_per_frame else chroma_tables(fs, K)
    cols = []
    Xp = None
    fv_prev = None
    pos = 0
    while pos + window - 1 < n:
        x = y[pos:pos + window]
        pos += step
        X = _spectrum(x, K)
        if Xp is None:
            Xp = X.copy()
        fv = np.zeros(N_BASE)
        fv[0] = _zcr(x)
        fv[1] = _energy(x)
        fv[2] = _block_entropy(x)
        fv[3], fv[4] = _centroid_spread(X, fs)
        fv[5] = _block_entropy(X)
        fv[6] = _flux(X, Xp)
        fv[7] = _rolloff(X, 0.90)
        fv[8:21] = dmat @ np.log10(bank @ X + EPS)                 # :252-253
        chroma = _chroma_frame(X, fs, K, fixed_tabs)
        fv[21:33] = chroma
        fv[33] = chroma.std()                                       # :667
        if deltas:
            d = np.zeros(N_BASE) if fv_prev is None else fv - fv_prev   # :672-678
            cols.append(np.concatenate([fv, d]))
            fv_prev = fv
        else:
            cols.append(fv)
        Xp = X
    if not cols:
        raise ValueError("need at least one array to concatenate")  # what :684 raises
    return np.stack(cols, axis=1), feature_names(deltas)


# --------------------------------------------------------------------------- vectorised flavour
def _frames_view(y, window, step, first, count):
    idx = first + step * np.arange(count)[:, None] + np.arange(window)[None, :]
    return y[idx]


def _spectra(frames, n_bins):
    return np.abs(np.fft.fft(frames, axis=1))[:, :n_bins] / n_bins


def _block_entropy_rows(V, n_blocks=10):
    total = np.sum(V ** 2, axis=1)
    blk = V.shape[1] // n_blocks
    parts = V[:, :blk * n_blocks].reshape(V.shape[0], n_blocks, blk)
    s = np.sum(parts ** 2, axis=2) / (total[:, None] + EPS)
    return -np.sum(s * np.log2(s + EPS), axis=1)


def base_features_from_frames(frames, X, fs):
    """All 34 base rows for a block of frames (rows) with spectra X; flux uses row t-1 (row 0: itself)."""
    T, w = frames.shape
    K = X.shape[1]
    out = np.zeros((N_BASE, T))
    out[0] = np.sum(np.abs(np.diff(np.sign(frames), axis=1)), axis=1) / 2 / np.float64(w - 1.0)
    out[1] = np.sum(frames ** 2, axis=1) / np.float64(w)
    out[2] = _block_entropy_rows(frames)
    ind = np.arange(1, K + 1) * (fs / (2.0 * K))
    top = X.max(axis=1)
    Xt = X / np.where(top == 0, EPS, top)[:, None]
    den = Xt.sum(axis=1) + EPS
    cen = (Xt * ind).sum(axis=1) / den
    spr = np.sqrt((((ind[None, :] - cen[:, None]) ** 2) * Xt).sum(axis=1) / den)
    out[3] = cen / (fs / 2.0)
    out[4] = spr / (fs / 2.0)
    out[5] = _block_entropy_rows(X)
    Xn = X / np.sum(X + EPS, axis=1)[:, None]
    prev = np.vstack([Xn[:1], Xn[:-1]])
    out[6] = np.sum((Xn - prev) ** 2, axis=1)
    P = X ** 2
    e = P.sum(axis=1)
    over = (np.cumsum(P, axis=1) + EPS) > (0.90 * e)[:, None]
    first = np.argmax(over, axis=1)
    out[7] = np.where(over.any(axis=1), first / float(K), 0.0)
    out[8:21] = dct_matrix() @ np.log10(mel_filterbank(fs, K) @ X.T + EPS)
    chroma = chroma_operator(fs, K) @ P.T
    chroma = chroma / np.where(e == 0, EPS, e)[None, :]
    out[21:33] = chroma
    out[33] = chroma.std(axis=0)
    return out


def feature_extraction(signal, fs, window, step, deltas=True):
    """Vectorised equivalent of ``feature_extraction_loop`` (ShortTermFeatures.py:543-685)."""
    window, step = int(window), int(step)
    y = normalize_clip(signal)
    T = frame_count(len(y), window, step)
    K = int(window / 2)
    mel_filterbank(fs, K)   # :578 -- built before the frame loop: its IndexError (:230-231) comes first
    if T == 0:
        raise ValueError("need at least one array to concatenate")          # :684
    chroma_operator(fs, K)  # raises early like the reference would on frame 0 (:290-294)
    rows = []
    chunk = max(1, (1 << 22) // window)
    Xlast = None
    for t0 in range(0, T, chunk):
        cnt = min(chunk, T - t0)
        lead = 1 if t0 > 0 else 0              # one frame of history for flux
        fr = _frames_view(y, window, step, (t0 - lead) * step, cnt + lead)
        X = _spectra(fr, K)
        rows.append(base_features_from_frames(fr, X, fs)[:, lead:])
    base = np.concatenate(rows, axis=1)
    if not deltas:
        return base, feature_names(False)
    delta = np.zeros_like(base)
    delta[:, 1:] = base[:, 1:] - base[:, :-1]
    return np.concatenate([base, delta], axis=0), feature_names(True)


def spectrogram(signal, fs, window, step):
    """ShortTermFeatures.py:389-452 without the plot / print side effects.

    Rows allocated ``int((N-w)/s)+1`` (:413); the loop starts at ``cur_p =
    window`` (:415), so row i is the spectrum of y[w+i*s : 2w+i*s] and the last
    rows stay zero.
    """
    window, step = int(window), int(step)
    y = normalize_clip(signal)
    n = len(y)
    K = int(window / 2)
    n_rows = int((n - window) / step) + 1
    spec = np.zeros((n_rows, K))
    starts = list(range(window, n - window + 1, step))
    if starts:
        fr = _frames_view(y, window, step, window, len(starts))
        spec[:len(starts)] = _spectra(fr, K)
    freq_axis = [float((f + 1) * fs) / (2 * K) for f in range(K)]
    time_axis = [float(t * step) / fs for t in range(n_rows)]
    return spec, time_axis, freq_axis


def chromagram(signal, fs, window, step):
    """ShortTermFeatures.py:324-386 without plotting.

    Rows ``int((N-s-w)/s)+1`` (:347), loop ``range(w, N-s, s)`` (:349): the
    last frame may be clipped at the end of the clip (shorter FFT, still
    ``[0:K]/K``), or the last row may stay zero.
    """
    window, step = int(window), int(step)
    y = normalize_clip(signal)
    n = len(y)
    K = int(window / 2)
    n_rows = int((n - step - window) / step) + 1
    out = np.zeros((n_rows, 12))
    op = chroma_operator(fs, K)
    for i, p in enumerate(range(window, n - step, step)):
        x = y[p:p + window]
        X = np.abs(np.fft.fft(x))[0:K]
        X = X / len(X)
        if len(X) != K:
            raise ValueError("shape mismatch: clipped last frame shorter than num_fft")
        P = X ** 2
        tot = P.sum()
        out[i, :] = (op @ P) / (EPS if tot == 0 else tot)
    time_axis = [(t * step) / fs for t in range(n_rows)]
    return out, time_axis, list(CHROMA_NAMES)


# --------------------------------------------------------------------------- mid-term pooling
def mid_ratios(mid_window, mid_step, short_window, short_step):
    """MidTermFeatures.py:100-102 (Python round = half-to-even)."""
    ratio = round((mid_window - (short_window - short_step)) / short_step)
    stepr = int(round(mid_step / short_step))
    return int(ratio), stepr


def mid_pool(short_features, ratio: int, stepr: int):
    """MidTermFeatures.py:110-126: mean / population std over sliding runs of st frames."""
    F, T = short_features.shape
    starts = list(range(0, T, stepr))
    mid = np.zeros((2 * F, len(starts)))
    for j, c in enumerate(starts):
        seg = short_features[:, c:min(c + ratio, T)]
        mid[:F, j] = seg.mean(axis=1)
        mid[F:, j] = seg.std(axis=1)
    return np.nan_to_num(mid)


def mid_feature_extraction(signal, fs, mid_window, mid_step, short_window, short_step, loop=False):
    """MidTermFeatures.py:87-127."""
    fe = feature_extraction_loop if loop else feature_extraction
    st, names = fe(signal, fs, short_window, short_step)
    ratio, stepr = mid_ratios(mid_window, mid_step, short_window, short_step)
    return mid_pool(st, ratio, stepr), st, mid_feature_names(names)


# --------------------------------------------------------------------------- synthetic clips (SURVEY 8d)
def synth_clip(index: int, n_samples: int = 160000, fs: int = 16000) -> np.ndarray:
    """Seeded int16 test clip: noise + three harmonics of a per-clip f0 (same recipe everywhere)."""
    rng = np.random.default_rng(1234 + int(index))
    f0 = rng.uniform(80.0, 1000.0)
    t = np.arange(n_samples) / float(fs)
    sig = 3000.0 * rng.standard_normal(n_samples)
    for h in (1, 2, 3):
        sig += 6000.0 * np.sin(2 * np.pi * h * f0 * t) / h
    return np.round(np.clip(sig, -32768, 32767)).astype(np.int16)
