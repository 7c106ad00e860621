"""GPU: everything after the short-term matrix against plain float64 restatements of the same operation.

- ``mid_pool_batch`` (mean / population std over runs of short-term frames, MidTermFeatures.py:110-126), across ratios,
  step ratios with overlaps and gaps, frame counts that clip the last window, ``n_frames`` below the row stride, and rows
  chosen where float accumulation, a one-pass variance or a float32 square would show.
- ``long_term_mean_batch`` (MidTermFeatures.py:200-201) up to 100 001 windows.
- ``normalize_windows_batch`` bit for bit against NumPy float32, with zero standard deviations, subnormals and more
  clips than one grid holds.
- The drop-in ``mid_feature_extraction``, the batched form and ``directory_feature_extraction`` end to end: they agree
  with each other bit for bit, pool the GPU's own short-term matrix to within one float32 ulp, and match the oracle.

The pooling kernels accumulate in float64 and round once to float32, so they are held to ``within_1ulp``.
"""
import warnings

import numpy as np
import pytest

from oracle import st_oracle as O
from tests.parity import check_features, check_mid, within_1ulp
from tests.test_oracle_vs_reference import CASES, case_setup

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def P():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import pyaudioanalysis_b200 as pkg
    pkg.MidTermFeatures.VERBOSE = False
    return pkg


def pool64(st, n_frames, ratio, stepr):
    """MidTermFeatures.py:110-124 in float64 over the first n_frames columns of a batch [B, F, >=n_frames] -> [B, 2F, M],
    before np.nan_to_num."""
    x = np.asarray(st)[:, :, :n_frames].astype(np.float64)
    B, F, _ = x.shape
    starts = range(0, n_frames, stepr)
    out = np.empty((B, 2 * F, len(starts)))
    with np.errstate(all="ignore"):
        for j, c in enumerate(starts):
            seg = x[:, :, c:min(c + ratio, n_frames)]
            out[:, :F, j] = seg.mean(axis=2)
            out[:, F:, j] = seg.std(axis=2)
    return out


def pool_ref(st, n_frames, ratio, stepr):
    """What the kernel must return: the float64 pooling rounded to float32, then np.nan_to_num (the kernel maps NaN to 0
    and +-inf to +-FLT_MAX after rounding)."""
    with np.errstate(all="ignore"):
        return np.nan_to_num(pool64(st, n_frames, ratio, stepr).astype(np.float32)).astype(np.float64)


# ------------------------------------------------------------------ mid_pool_batch
ROW_KINDS = ("const", "huge", "nan", "+inf", "-inf", "offset", "offset")


def pool_rows(rng, B, F, T, pad):
    """[B, F, T + pad] float32: row 0 is 3e4 + 0.05 N(0, 1) (float accumulation and a one-pass variance lose the spread to
    the offset), the others cycle through constant rows (std exactly 0), values near +-3e38 (float32 squares and sums
    overflow, float64 does not), one NaN / +inf / -inf in an offset row, and more offset rows.  Columns past T hold 1e30,
    so a read past n_frames shows."""
    x = np.full((B, F, T + pad), 1e30, dtype=np.float32)
    for r in range(B * F):
        b, f = divmod(r, F)
        kind = "offset" if r == 0 else ROW_KINDS[(r - 1) % len(ROW_KINDS)]
        if kind == "const":
            row = np.full(T, rng.normal() * 100.0)
        elif kind == "huge":
            row = rng.choice([-1.0, 1.0], T) * rng.uniform(2.9e38, 3.1e38, T)
        else:
            row = 3e4 + 0.05 * rng.standard_normal(T)
        row = row.astype(np.float32)
        if kind in ("nan", "+inf", "-inf"):
            row[rng.integers(T)] = {"nan": np.nan, "+inf": np.inf, "-inf": -np.inf}[kind]
        x[b, f, :T] = row
    return x


POOL_RATIOS = (1, 2, 31, 32, 33, 39, 64, 65, 1000)
STEP_KINDS = ("1", "r-1", "r", "r+7", "2r")


def _step_ratio(ratio, kind):
    return {"1": 1, "r-1": max(1, ratio - 1), "r": ratio, "r+7": ratio + 7, "2r": 2 * ratio}[kind]


@pytest.mark.parametrize("step_kind", STEP_KINDS)
@pytest.mark.parametrize("ratio", POOL_RATIOS)
def test_mid_pool_matrix(P, ratio, step_kind):
    """Every (B, F) in {1, 3} x {1, 33, 34, 68} at T = 1, T < ratio, T = ratio, T = 3 step ratios (whole last window or
    a clipped one) and 3 step ratios + 1 (a last window of one frame, whose std must be exactly 0)."""
    import torch
    from pyaudioanalysis_b200.batch import mid_pool_batch
    stepr = _step_ratio(ratio, step_kind)
    Ts = sorted({1, max(1, ratio // 2), ratio, 3 * stepr, 3 * stepr + 1})
    rng = np.random.default_rng(1000 * ratio + STEP_KINDS.index(step_kind))
    for T in Ts:
        for B in (1, 3):
            for F in (1, 33, 34, 68):
                pad = 0 if F == 34 else 5                    # n_frames == row stride, and n_frames < row stride
                st = pool_rows(rng, B, F, T, pad)
                mid = mid_pool_batch(torch.from_numpy(st).cuda(), ratio, stepr, n_frames=T if pad else None).cpu().numpy()
                M = -(-T // stepr)
                assert mid.shape == (B, 2 * F, M)
                within_1ulp(mid, pool_ref(st, T, ratio, stepr), "mid_pool ratio %d step %d T %d B %d F %d" % (ratio, stepr, T, B, F))
                if (T - 1) % stepr == 0:                     # last window holds one frame: std exactly 0
                    assert not mid[:, F:, -1].any()


def test_mid_pool_normal_rows_and_errors(P):
    """N(0, 1) rows at the reference's default 39 / 40 with T = 399 = row stride, plus the argument checks."""
    import torch
    from pyaudioanalysis_b200.batch import mid_pool_batch
    st = torch.randn(3, 68, 399, device="cuda")
    mid = mid_pool_batch(st, 39, 40).cpu().numpy()
    within_1ulp(mid, pool_ref(st.cpu().numpy(), 399, 39, 40), "mid_pool N(0, 1) 39 / 40")
    for ratio, stepr, n in ((0, 40, None), (-3, 40, None), (39, 0, None), (39, -1, None), (39, 40, 400), (39, 40, 0)):
        with pytest.raises(ValueError):
            mid_pool_batch(st, ratio, stepr, n_frames=n)


# ------------------------------------------------------------------ long_term_mean_batch
@pytest.mark.parametrize("M", (1, 2, 31, 32, 33, 3600, 100001))
def test_long_term_mean_matrix(P, M):
    """Rows of 50 + N(0, 1) (float accumulation over 100 001 windows is ~16 ulps off), of +-1e38 (a float sum
    overflows) and of zeros; rows in {1, 136, 138}, clips in {1, 5}."""
    import torch
    from pyaudioanalysis_b200.batch import long_term_mean_batch
    rng = np.random.default_rng(M)
    for B in (1, 5):
        for rows in (1, 136, 138):
            mid = (50.0 + rng.standard_normal((B, rows, M))).astype(np.float32)
            mid[:, 3::4] = (rng.choice([-1.0, 1.0], (B, mid[:, 3::4].shape[1], M)) * 1e38).astype(np.float32)
            mid[:, 5::7] = 0.0
            got = long_term_mean_batch(torch.from_numpy(mid).cuda()).cpu().numpy()
            assert got.shape == (B, rows)
            within_1ulp(got, mid.mean(axis=2, dtype=np.float64), "long_term_mean M %d rows %d B %d" % (M, rows, B))


# ------------------------------------------------------------------ normalize_windows_batch
def assert_same_bits(got, ref, what):
    """float32 arrays equal bit for bit; NaNs compared by position only."""
    assert got.shape == ref.shape and got.dtype == ref.dtype == np.float32, (what, got.shape, ref.shape)
    ng, nr = np.isnan(got), np.isnan(ref)
    assert (ng == nr).all(), "%s: NaN positions differ" % what
    diff = got[~ng].view(np.uint32) != ref[~nr].view(np.uint32)
    assert not diff.any(), "%s: %d of %d values differ in their bits" % (what, int(diff.sum()), diff.size)


def normalize_case(rng, B, F, M, kinds_shift=0):
    """mid [B, F, M] float32 and float64 mean / std [F].  Row kinds cycle: ordinary, subnormal values over a std of 0.75
    (subnormal results: flush-to-zero shows), zero std (+-inf, and NaN where the value equals the mean), ordinary."""
    mid = (rng.standard_normal((B, F, M)) * 7.0).astype(np.float32)
    mean = rng.standard_normal(F) * 3.0
    std = rng.uniform(0.5, 2.0, F)
    for f in range(F):
        kind = (f + kinds_shift) % 4
        if kind == 1:
            mid[:, f] = (rng.uniform(-1, 1, (B, M)) * 1e-39).astype(np.float32)
            mean[f], std[f] = 0.0, 0.75
        elif kind == 2:
            std[f] = 0.0
            mid[:, f, ::2] = np.float32(mean[f])
    return mid, mean, std


def normalize_ref(mid, mean, std):
    with np.errstate(all="ignore"):
        return ((mid - mean.astype(np.float32)[None, :, None]) / std.astype(np.float32)[None, :, None]).transpose(0, 2, 1)


@pytest.mark.parametrize("M", (1, 31, 32, 33, 3600))
@pytest.mark.parametrize("F", (1, 31, 32, 33, 136, 138))
def test_normalize_windows_matrix(P, F, M):
    import torch
    from pyaudioanalysis_b200.consumers import normalize_windows_batch
    rng = np.random.default_rng(F * 10007 + M)
    for B in (1, 3):
        mid, mean, std = normalize_case(rng, B, F, M, kinds_shift=M)
        out = normalize_windows_batch(torch.from_numpy(mid).cuda(), mean, std).cpu().numpy()
        assert_same_bits(out, normalize_ref(mid, mean, std), "normalize F %d M %d B %d" % (F, M, B))


def test_normalize_windows_shapes_and_errors(P):
    """Shapes of the classifier consumers (136 rows, 8 .. 399 windows, one window), 70 000 clips (more than the 65 535
    one grid holds) and a mean / std of the wrong length."""
    import torch
    from pyaudioanalysis_b200.consumers import normalize_windows_batch
    rng = np.random.default_rng(11)
    for B, F, M in ((1, 136, 8), (3, 136, 77), (2, 68, 399), (5, 7, 1), (1, 33, 65), (70000, 3, 2)):
        mid, mean, std = normalize_case(rng, B, F, M)
        out = normalize_windows_batch(torch.from_numpy(mid).cuda(), mean, std).cpu().numpy()
        assert out.shape == (B, M, F)
        assert_same_bits(out, normalize_ref(mid, mean, std), "normalize B %d F %d M %d" % (B, F, M))
    with pytest.raises(ValueError):
        normalize_windows_batch(torch.zeros((1, 4, 4), device="cuda"), np.zeros(3), np.ones(3))


# ------------------------------------------------------------------ mid-term end to end
def _extra(fs, w, s, n, mw, ms, seed):
    return {"fs": fs, "w": w, "s": s, "x": O.synth_clip(seed, n, fs), "mw": mw, "ms": ms}


def mid_cases():
    """(id, fs, w, s, clip, mid window, mid step): the randomised configurations the oracle is pinned to the reference on
    (tests/test_oracle_vs_reference.py, float64 inputs with a DC offset among them) and the shapes of common use."""
    out = []
    for i, (fs, w, s, n, seed) in enumerate(CASES):
        x, mw, ms = case_setup(fs, w, s, n, seed)
        out.append(("case%d" % i, fs, w, s, x, mw, ms))
    out += [
        ("16k_39_40", 16000, 800, 400, O.synth_clip(501, 5 * 16000 + 123, 16000), 16000, 16000),
        ("800_800_10_2", 16000, 800, 800, O.synth_clip(502, 3 * 16000, 16000), 0.5 * 16000, 0.1 * 16000),
        ("44k_199_100", 44100, 882, 441, O.synth_clip(503, 5 * 44100 + 7, 44100), 2.0 * 44100, 1.0 * 44100),
        ("shorter_than_mid", 16000, 800, 400, O.synth_clip(504, 6000, 16000), 16000, 16000),
        ("T1", 16000, 800, 400, O.synth_clip(505, 800, 16000), 16000, 16000),
        ("T81", 16000, 800, 400, O.synth_clip(506, 32800, 16000), 16000, 16000),
        ("chroma_error", 8000, 160, 80, O.synth_clip(507, 1000, 8000), 640, 640),      # ValueError at frame 0
        ("mel_error", 4000, 100, 50, O.synth_clip(508, 1000, 4000), 400, 400),         # IndexError building the mel bank
    ]
    return out


MID_CASES = mid_cases()


def _as_int16(x):
    return x if x.dtype == np.int16 else np.round(np.clip(x, -32768, 32767)).astype(np.int16)


def _as_float(x):
    return x if x.dtype != np.int16 else x.astype(np.float64) * 0.37 + 11.5


@pytest.mark.parametrize("kind", ("int16", "float"))
@pytest.mark.parametrize("case", MID_CASES, ids=[c[0] for c in MID_CASES])
def test_mid_feature_extraction_end_to_end(P, case, kind):
    """Drop-in call == batched call on 3 distinct clips (bit for bit); the mid matrix within one ulp of pooling the
    GPU's own short-term matrix; short-term rows within the standard tolerance of the oracle and mid-term rows within the
    propagated one.  Where the oracle raises, the GPU raises the same type."""
    import torch
    from pyaudioanalysis_b200.batch import mid_feature_extraction_batch, mid_ratios
    _, fs, w, s, x, mw, ms = case
    x = _as_int16(x) if kind == "int16" else _as_float(x)
    clips = [x, np.roll(x, 1234), x[::-1].copy()]
    try:
        ref_mid, ref_st, ref_names = O.mid_feature_extraction(x, fs, mw, ms, w, s)
    except (ValueError, IndexError) as e:
        with pytest.raises(type(e)):
            P.MidTermFeatures.mid_feature_extraction(x, fs, mw, ms, w, s)
        dev = torch.from_numpy(np.stack(clips).astype(np.int16 if kind == "int16" else np.float32)).cuda()
        with pytest.raises(type(e)):
            mid_feature_extraction_batch(dev, fs, mw, ms, w, s)
        return
    drop = [P.MidTermFeatures.mid_feature_extraction(c, fs, mw, ms, w, s) for c in clips]
    assert drop[0][2] == ref_names
    dev = torch.from_numpy(np.stack(clips).astype(np.int16 if kind == "int16" else np.float32)).cuda()
    mid_b, st_b = mid_feature_extraction_batch(dev, fs, mw, ms, w, s)
    mid_b, st_b = mid_b.cpu().numpy(), st_b.cpu().numpy()
    for k in range(3):
        assert np.array_equal(drop[k][0].astype(np.float32), mid_b[k]), "clip %d: drop-in and batched mid-term differ" % k
        assert np.array_equal(drop[k][1].astype(np.float32), st_b[k]), "clip %d: drop-in and batched short-term differ" % k
    ratio, stepr = mid_ratios(mw, ms, w, s)
    within_1ulp(mid_b, pool_ref(st_b, st_b.shape[2], ratio, stepr), "pooling of the GPU short-term matrix")
    check_features(drop[0][1], ref_st, w // 2, "short-term")
    check_mid(drop[0][0], ref_mid, ref_st, "mid-term")


def test_mid_ratio_below_one_diverges(P):
    """The one known divergence from the reference: a mid-term window shorter than one short-term step (ratio < 1).
    The GPU raises ValueError.  The reference pools empty slices for ratio 0 (all-zero output after np.nan_to_num) and,
    for ratio < 0, Python slices st[:, c:c + ratio] that end `ratio` frames before the end of the clip."""
    import torch
    from pyaudioanalysis_b200.batch import mid_feature_extraction_batch
    fs, w, s = 16000, 800, 400
    x = O.synth_clip(510, 16000, fs)
    for mw, ratio in ((200, 0), (-800, -3)):
        assert O.mid_ratios(mw, 8000, w, s) == (ratio, 20)
        with pytest.raises(ValueError):
            P.MidTermFeatures.mid_feature_extraction(x, fs, mw, 8000, w, s)
        with pytest.raises(ValueError):
            mid_feature_extraction_batch(torch.from_numpy(x).cuda(), fs, mw, 8000, w, s)
        with warnings.catch_warnings():                 # NumPy warns about the empty slices of ratio 0
            warnings.simplefilter("ignore", RuntimeWarning)
            rm, rs, _ = O.mid_feature_extraction(x, fs, mw, 8000, w, s)
        if ratio == 0:
            assert not rm.any()
        else:
            np.testing.assert_allclose(rm[:68, 0], rs[:, :rs.shape[1] + ratio].mean(axis=1), rtol=1e-12)


def test_directory_long_term_means(P, tmp_path):
    """directory_feature_extraction(compute_beat=False) on files at 8 and 16 kHz, of three lengths of 3 s or more (so
    several mid-term windows), one of them stereo and one float32: sorted file order, every row within one ulp of the
    float64 mean of the drop-in mid-term matrix of its file, and within the propagated tolerance of the oracle."""
    from scipy.io import wavfile
    from pyaudioanalysis_b200 import audioio
    files = {
        "b_16k.wav": (16000, O.synth_clip(601, 48000, 16000)),
        "A_8k.wav": (8000, O.synth_clip(602, 36000, 8000)),
        "c_stereo.wav": (16000, np.stack([O.synth_clip(603, 56000, 16000), O.synth_clip(604, 56000, 16000)], axis=1)),
        "a_float.wav": (16000, (O.synth_clip(605, 48000, 16000) / 32768.0 * 0.8).astype(np.float32)),
        "d_16k.wav": (16000, O.synth_clip(606, 48000, 16000)),
        "e_8k.wav": (8000, O.synth_clip(607, 24000, 8000)),
    }
    for name, (fs, x) in files.items():
        wavfile.write(str(tmp_path / name), fs, x)
    mt_w, mt_s, st_w, st_s = 1.0, 0.5, 0.05, 0.025
    feats, got_files, names = P.MidTermFeatures.directory_feature_extraction(str(tmp_path), mt_w, mt_s, st_w, st_s,
                                                                            compute_beat=False)
    assert [f.split("/")[-1] for f in got_files] == sorted(files)
    assert feats.shape == (len(files), 136) and len(names) == 136
    for row, path in zip(feats, got_files):
        fs, x = audioio.read_audio_file(path)
        x = audioio.stereo_to_mono(x)
        args = (fs, round(mt_w * fs), round(mt_s * fs), round(fs * st_w), round(fs * st_s))
        mid, _, _ = P.MidTermFeatures.mid_feature_extraction(x, *args)
        assert mid.shape[1] > 1
        within_1ulp(row, mid.mean(axis=1), "long-term mean of " + path)
        ref_mid, ref_st, _ = O.mid_feature_extraction(x, *args)
        check_mid(row[:, None], ref_mid.mean(axis=1)[:, None], ref_st, "directory row of " + path)
