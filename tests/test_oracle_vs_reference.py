"""CPU: the oracle against values of the UNMODIFIED reference on randomised configurations, its tables and its error cases.

The reference's outputs are stored in tests/golden/vs_reference.npz (oracle/make_golden_vs_reference.py).  A matrix is
held to the reference through its shape, its sums along the last axis and a seeded sample of its elements.
"""
import numpy as np
import pytest

from oracle import st_oracle as O
from tests.conftest import load_golden

EXCEPTIONS = {"ValueError": ValueError, "IndexError": IndexError}

CASES = []
_rng = np.random.default_rng(20260922)
for _ in range(14):
    fs = int(_rng.choice([8000, 16000, 22050, 32000, 44100, 48000]))
    w = int(_rng.integers(max(240, fs // 70), fs // 12))
    s = int(_rng.integers(max(1, w // 8), w + 1))
    n = int(_rng.integers(3 * w, 12 * w))
    CASES.append((fs, w, s, n, int(_rng.integers(0, 10 ** 6))))

TABLE_CASES = [(16000, 400), (44100, 441), (8000, 200), (22050, 551), (48000, 1200)]
ERROR_CASES = [(4000, 100, 50, 50), (4000, 100, 50, 1000), (8000, 160, 80, 100), (8000, 160, 80, 1000), (4000, 400, 200, 100),
               (16000, 800, 400, 799)]


@pytest.fixture(scope="module")
def REF():
    g = dict(load_golden("vs_reference.npz"))
    assert g["cases"].tolist() == [list(c) for c in CASES], "golden values were made for other configurations"
    counts, rows = g["sum_counts"], g["sum_shapes"][:, 0]
    so, ro = np.concatenate([[0], np.cumsum(counts)]), np.concatenate([[0], np.cumsum(rows)])
    for i, key in enumerate(g["sum_keys"].tolist()):        # unpack oracle/make_golden_vs_reference.py's summaries
        g[key] = (tuple(g["sum_shapes"][i]), g["sum_idx"][so[i]:so[i + 1]], g["sum_val"][so[i]:so[i + 1]], g["sum_rowsum"][ro[i]:ro[i + 1]])
    return g


def case_setup(fs, w, s, n, seed):
    """The clip of one configuration and its mid-term window / step (one generator per case, drawn in this order)."""
    rng = np.random.default_rng(seed)
    x = O.synth_clip(seed, n, fs)
    if seed % 3 == 0:                       # float-valued input with a DC offset
        x = x.astype(np.float64) * float(rng.uniform(0.01, 3.0)) + float(rng.uniform(-500, 500))
    mw, ms = int(rng.integers(2, 9)) * s + w, int(rng.integers(1, 9)) * s
    return x, mw, ms


def match(got, g, key, rtol, atol):
    """Same shape as the reference's output `key` (a 1-D output is one row), its sampled elements within rtol / atol, and
    every sum along the last axis within the bound that elementwise closeness implies."""
    shape, idx, val, rowsum = g[key]
    got = np.atleast_2d(np.asarray(got, dtype=np.float64))
    assert got.shape == shape, (key, got.shape, shape)
    np.testing.assert_allclose(got.reshape(-1)[idx], val, rtol=rtol, atol=atol, err_msg=key)
    bound = rtol * np.abs(got).sum(axis=-1) + atol * got.shape[-1]
    assert np.all(np.abs(got.sum(axis=-1) - rowsum) <= bound), key


@pytest.mark.parametrize("fs,w,s,n,seed", CASES)
def test_random_configurations(REF, fs, w, s, n, seed):
    k = "case%d" % CASES.index((fs, w, s, n, seed))
    x, mw, ms = case_setup(fs, w, s, n, seed)
    deltas = bool(seed % 2)
    if k + "_exc" in REF:
        with pytest.raises(EXCEPTIONS[str(REF[k + "_exc"])]):
            O.feature_extraction(x, fs, w, s, deltas=deltas)
        return
    got, gnames = O.feature_extraction(x, fs, w, s, deltas=deltas)
    assert gnames == list(REF["names_deltas%d" % deltas])
    match(got, REF, k + "_st", 1e-8, 1e-10)
    loop, _ = O.feature_extraction_loop(x[: 4 * w], fs, w, s, deltas=deltas)
    match(loop, REF, k + "_loop", 1e-8, 1e-10)
    sp = O.spectrogram(x, fs, w, s)
    match(sp[0], REF, k + "_sp", 1e-9, 1e-12)
    match(sp[1], REF, k + "_sp_time", 0, 0)
    match(sp[2], REF, k + "_sp_freq", 0, 0)
    if k + "_ch_exc" in REF:
        with pytest.raises(ValueError):
            O.chromagram(x, fs, w, s)
    else:
        ch = O.chromagram(x, fs, w, s)
        match(ch[0], REF, k + "_ch", 1e-9, 1e-12)
        match(ch[1], REF, k + "_ch_time", 0, 0)
        assert ch[2] == list(REF["chroma_names"])
    mid = O.mid_feature_extraction(x, fs, mw, ms, w, s)
    match(mid[0], REF, k + "_mid", 1e-8, 1e-10)
    assert mid[2] == list(REF["mid_names"])


def test_tables_match_reference(REF):
    for fs, K in TABLE_CASES:
        k = "tab_%d_%d" % (fs, K)
        np.testing.assert_array_equal(O.mel_filterbank(fs, K), REF[k + "_mel"])
        os_, osh = O.chroma_tables(fs, K)
        np.testing.assert_array_equal(os_, REF[k + "_semis"])
        np.testing.assert_array_equal(osh, REF[k + "_share"])
        X = np.random.default_rng(K).random(K)
        np.testing.assert_allclose(O.chroma_operator(fs, K) @ (X ** 2) / (X ** 2).sum(), REF[k + "_chroma"], rtol=1e-12, atol=1e-15)


@pytest.mark.parametrize("fs,w,s,n", ERROR_CASES)
def test_error_precedence(REF, fs, w, s, n):
    """mel bank IndexError (before the loop) > no frames ValueError > chroma ValueError (frame 0)."""
    k = "err_%d_%d_%d_%d" % (fs, w, s, n)
    exc = EXCEPTIONS[str(REF[k + "_exc"])]
    x = O.synth_clip(1, n, fs)
    with pytest.raises(exc) as got:
        O.feature_extraction(x, fs, w, s)
    assert ("need at least one array" in str(got.value)) == bool(REF[k + "_no_frames"])
    with pytest.raises(exc):
        O.feature_extraction_loop(x, fs, w, s)
