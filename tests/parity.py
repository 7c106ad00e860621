"""Shared comparison helpers for the GPU parity tests.

Tolerance (stated once, used everywhere): every feature column must satisfy
    |gpu - ref| <= RTOL * |ref| + ATOL      with RTOL = 1e-4, ATOL = 1e-5
(BASELINE.json north_star asks for 1e-4 rtol; the absolute term covers values that cross zero --
mfcc_2..13 and every delta column are differences of near-equal numbers -- see SURVEY.md 8d.)
Two rows are discrete: zcr moves in quanta of 0.5/(w-1) and spectral_rolloff in quanta of 1/K; a
float32-vs-float64 tie may move them by one quantum on a small fraction of frames, which is
counted and bounded separately.

Mid-term rows (means / standard deviations over runs of short-term frames) inherit the short-term tolerance scaled to
each short-term row's magnitude: a standard deviation of nearly constant values carries the ABSOLUTE error of its
inputs, and one rolloff quantum flip moves that window's rolloff mean and std, so ``check_mid`` skips the four rolloff
rows.  The pooling itself is held to ``within_1ulp``: the kernels accumulate in float64 and round once to float32.
"""
import numpy as np

RTOL, ATOL = 1e-4, 1e-5
ROLLOFF_ROW = 7
MAX_FLIP_FRACTION = 2e-3


def check_features(gpu, ref, K, what=""):
    gpu = np.asarray(gpu, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert gpu.shape == ref.shape, (what, gpu.shape, ref.shape)
    assert np.isfinite(gpu).all(), what + ": non-finite output"
    err = np.abs(gpu - ref)
    tol = RTOL * np.abs(ref) + ATOL
    bad = err > tol
    F = ref.shape[0]
    flips = 0
    for r in (ROLLOFF_ROW, ROLLOFF_ROW + 34):
        if r < F and bad[r].any():
            q = err[r][bad[r]]
            assert (q <= (1.0 / K) * (2 if r >= 34 else 1) + 1e-6).all(), "%s: rolloff off by more than one quantum" % what
            flips += int(bad[r].sum())
            bad[r] = False
    assert flips <= max(2, MAX_FLIP_FRACTION * ref.shape[1] * 2), "%s: %d rolloff quantum flips" % (what, flips)
    if bad.any():
        rows = np.unique(np.nonzero(bad)[0])
        worst = [(int(r), float(err[r].max()), float((err[r] / tol[r]).max())) for r in rows]
        raise AssertionError("%s: rows outside tolerance (row, max abs err, max err/tol): %s" % (what, worst))
    return flips


def check_close(gpu, ref, what="", rtol=RTOL, atol=ATOL):
    gpu = np.asarray(gpu, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert gpu.shape == ref.shape, (what, gpu.shape, ref.shape)
    np.testing.assert_allclose(gpu, ref, rtol=rtol, atol=atol, err_msg=what)


MID_ROLLOFF_ROWS = (ROLLOFF_ROW, ROLLOFF_ROW + 34, 68 + ROLLOFF_ROW, 68 + ROLLOFF_ROW + 34)


def check_mid(gpu, ref_mid, ref_st, what=""):
    """GPU mid-term matrix [2F x M] against the reference's, given the reference's short-term matrix [F x T]:
    |gpu - ref| <= 1e-4 * max|short-term row| + 1e-5 + 1e-4 * |ref| on every row except the rolloff rows."""
    gpu = np.asarray(gpu, dtype=np.float64)
    ref_mid = np.asarray(ref_mid, dtype=np.float64)
    assert gpu.shape == ref_mid.shape, (what, gpu.shape, ref_mid.shape)
    assert np.isfinite(gpu).all(), what + ": non-finite output"
    n_rows = ref_mid.shape[0]
    keep = np.ones(n_rows, bool)
    keep[[r for r in MID_ROLLOFF_ROWS if r < n_rows]] = False
    scale = np.abs(np.asarray(ref_st, dtype=np.float64)).max(axis=1)      # per short-term row
    tol = RTOL * np.concatenate([scale, scale])[:, None] + ATOL + RTOL * np.abs(ref_mid)
    bad = (np.abs(gpu - ref_mid) > tol) & keep[:, None]
    assert not bad.any(), "%s: mid-term rows outside tolerance: %s" % (what, np.unique(np.nonzero(bad)[0]).tolist())


def within_1ulp(gpu, ref64, what=""):
    """Elementwise |gpu - ref64| <= one float32 ulp of |ref64|, and exactly 0 where ref64 is 0: the bar for a kernel that
    computes in float64 and rounds once to float32 (a correctly rounded result is within half an ulp of the exact value;
    a different float64 summation order may move a tie by one ulp)."""
    gpu = np.asarray(gpu)
    ref64 = np.asarray(ref64, dtype=np.float64)
    assert gpu.shape == ref64.shape, (what, gpu.shape, ref64.shape)
    g = gpu.astype(np.float64)
    assert np.isfinite(g).all() and np.isfinite(ref64).all(), what + ": non-finite values"
    zero = ref64 == 0
    assert (g[zero] == 0).all(), "%s: %d entries should be exactly 0" % (what, int((g[zero] != 0).sum()))
    a = np.abs(ref64).astype(np.float32)
    with np.errstate(over="ignore"):
        up = np.spacing(a)
    ulp = np.where(np.isinf(up), a - np.nextafter(a, np.float32(0)), up).astype(np.float64)   # FLT_MAX: the gap below
    err = np.abs(g - ref64)
    bad = (err > ulp) & ~zero
    if bad.any():
        i = np.unravel_index(np.argmax(np.where(bad, err / ulp, 0)), bad.shape)
        raise AssertionError("%s: %d entries more than 1 ulp off; worst at %s: gpu %r, ref %r (%.1f ulp)"
                             % (what, int(bad.sum()), tuple(int(k) for k in i), float(g[i]), float(ref64[i]), float(err[i] / ulp[i])))
