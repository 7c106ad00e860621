"""Golden values for tests/test_oracle_vs_reference.py from the UNMODIFIED reference (run where the reference tree exists):

    python -m oracle.make_golden_vs_reference

For the test's randomised configurations, the reference's feature_extraction (also on a 4-window prefix), spectrogram,
chromagram and mid_feature_extraction are reduced to what the test needs to hold the oracle to them: the shape, the
sums along the last axis (every element enters one) and a seeded sample of 32 elements with their flat positions
(``summary``, packed into a few arrays by ``pack``).  Exceptions are stored by type name.  The filter-bank / chroma tables are small and stored whole, as are
the exception types of the error-precedence cases.  Writes tests/golden/vs_reference.npz.
"""
import contextlib
import io
import os

import numpy as np

from oracle import st_oracle as O
from oracle.ref_import import load_reference
from tests.test_oracle_vs_reference import CASES, ERROR_CASES, TABLE_CASES, case_setup

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "vs_reference.npz")
SAMPLE = 32


def summary(out, key, a, seed):
    """Shape, sums along the last axis and a seeded sample of the elements of `a` (1-D as one row), kept for `pack`."""
    a = np.atleast_2d(np.asarray(a, dtype=np.float64))
    idx = np.sort(np.random.default_rng(seed).choice(a.size, min(SAMPLE, a.size), replace=False))
    out.setdefault("summaries", []).append((key, a.shape, idx, a.reshape(-1)[idx], a.sum(axis=-1)))


def pack(summaries):
    """All summaries as six arrays (one .npy each keeps the file small); tests/test_oracle_vs_reference.py unpacks them."""
    keys, shapes, idx, val, rowsum = zip(*summaries)
    return {"sum_keys": np.array(keys), "sum_shapes": np.array(shapes, dtype=np.int64),
            "sum_counts": np.array([len(i) for i in idx], dtype=np.int64), "sum_idx": np.concatenate(idx).astype(np.int64),
            "sum_val": np.concatenate(val), "sum_rowsum": np.concatenate(rowsum)}


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def main():
    S, M, A = load_reference()
    out = {"cases": np.array(CASES, dtype=np.int64)}
    for i, (fs, w, s, n, seed) in enumerate(CASES):
        k = "case%d" % i
        x, mw, ms = case_setup(fs, w, s, n, seed)
        deltas = bool(seed % 2)
        try:
            ref, names = S.feature_extraction(x, fs, w, s, deltas=deltas)
        except (ValueError, IndexError) as exc:
            out[k + "_exc"] = np.array(type(exc).__name__)
            continue
        out["names_deltas%d" % deltas] = np.array(names)
        summary(out, k + "_st", ref, seed)
        summary(out, k + "_loop", S.feature_extraction(x[: 4 * w], fs, w, s, deltas=deltas)[0], seed + 1)
        sp = quiet(S.spectrogram, x, fs, w, s)
        summary(out, k + "_sp", sp[0], seed + 2)
        summary(out, k + "_sp_time", sp[1], seed + 3)
        summary(out, k + "_sp_freq", sp[2], seed + 4)
        try:
            ch = S.chromagram(x, fs, w, s)
        except ValueError:
            out[k + "_ch_exc"] = np.array("ValueError")
        else:
            summary(out, k + "_ch", ch[0], seed + 5)
            summary(out, k + "_ch_time", ch[1], seed + 6)
            out["chroma_names"] = np.array(ch[2])
        mid = M.mid_feature_extraction(x, fs, mw, ms, w, s)
        summary(out, k + "_mid", mid[0], seed + 7)
        out["mid_names"] = np.array(mid[2])
    for fs, K in TABLE_CASES:
        k = "tab_%d_%d" % (fs, K)
        out[k + "_mel"] = S.mfcc_filter_banks(fs, K)[0]
        out[k + "_semis"], out[k + "_share"] = S.chroma_features_init(K, fs)
        X = np.random.default_rng(K).random(K)
        out[k + "_chroma"] = S.chroma_features(X, fs, K)[1][:, 0]
    for fs, w, s, n in ERROR_CASES:
        k = "err_%d_%d_%d_%d" % (fs, w, s, n)
        try:
            S.feature_extraction(O.synth_clip(1, n, fs), fs, w, s)
        except (ValueError, IndexError) as exc:
            out[k + "_exc"] = np.array(type(exc).__name__)
            out[k + "_no_frames"] = np.array("need at least one array" in str(exc))
        else:
            raise AssertionError("the reference no longer raises on %s" % k)
    out.update(pack(out.pop("summaries")))
    np.savez_compressed(OUT, **out)
    print(OUT, os.path.getsize(OUT))


if __name__ == "__main__":
    main()
