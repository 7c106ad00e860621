"""GPU: the batched normalise-and-classify consumers (pyaudioanalysis_b200/consumers.py, b200aa_normalize_windows) against
the reference's per-window loops restated on the oracle's float64 mid-term matrix (audioSegmentation.py:571-591,
audioTrainTest.py:1074-1095)."""
import types

import numpy as np
import pytest

from oracle import st_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def P():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import pyaudioanalysis_b200 as pkg
    return pkg


def test_mid_term_classification_matches_reference_loop(P):
    """Windows of a two-part clip (noise, then a tone) through mid features -> normalise -> SVM / kNN: labels and maximum
    posteriors of the batched path equal the reference's per-window loop run on the oracle's float64 matrix."""
    from sklearn.svm import SVC
    from pyaudioanalysis_b200 import consumers as C
    fs = 16000
    rng = np.random.default_rng(5)
    t = np.arange(6 * fs)
    x = np.concatenate([rng.normal(0, 3000, 6 * fs), 9000 * np.sin(2 * np.pi * 440 * t / fs) + rng.normal(0, 300, 6 * fs)])
    x = np.round(np.clip(x, -32768, 32767)).astype(np.int16)
    mt, st = 1.0, 0.05
    ref_mid, _, _ = O.mid_feature_extraction(x, fs, mt * fs, mt * fs, round(fs * st), round(fs * st))
    M = ref_mid.shape[1]
    mean, std = ref_mid.mean(axis=1), ref_mid.std(axis=1) + 1e-3
    Xn = ((ref_mid - mean[:, None]) / std[:, None]).T
    y = (np.arange(M) >= M // 2).astype(int)
    svm = SVC(C=1.0, kernel="linear", probability=True, random_state=0).fit(Xn, y)
    knn = types.SimpleNamespace(features=Xn, labels=y, neighbors=3)
    for clf, kind in ((svm, "svm"), (knn, "knn")):
        labels, post = C.mid_term_classification(x, fs, clf, kind, mean, std, mt, mt, st, st)
        ref_labels, ref_post = [], []
        for j in range(M):                                  # audioSegmentation.py:579-590
            v = (ref_mid[:, j] - mean) / std
            if kind == "knn":
                i, p = C.knn_classify_matrix(clf, v.reshape(1, -1))
                i, p = i[0], p[0]
            else:
                i, p = clf.predict(v.reshape(1, -1))[0], clf.predict_proba(v.reshape(1, -1))[0]
            ref_labels.append(i)
            ref_post.append(np.max(p))
        assert list(labels) == ref_labels, kind
        assert np.allclose(post, ref_post, rtol=1e-3, atol=1e-3), kind
    segs, classes = C.labels_to_segments(labels, mt)
    assert list(classes) == [0, 1] and segs[0][1] == M // 2 * mt
    # file-level vector (audioTrainTest.py:1084-1095): long-term average (+ beat), normalised, classified
    lt = ref_mid.mean(axis=1)
    cid, prob = C.file_classification_vector(x, fs, svm, "svm", mean, std, mt, mt, st, st)
    v = ((lt - mean) / std).reshape(1, -1)
    assert cid == svm.predict(v)[0] and np.allclose(prob, svm.predict_proba(v)[0], rtol=1e-3, atol=1e-3)
