"""GPU parity at the sizes BASELINE.json names (configs[2], [3], [4]), against the oracle.

configs[1] at size is test_gpu_parity.py::test_full_size_properties.  Inputs are seeded on the host so the oracle
sees bit-identical samples; the oracle handles these sizes in seconds (vectorised flavour, chunked over frames).
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import st_oracle as O
from tests.parity import check_features, check_close, check_mid

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def P():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import pyaudioanalysis_b200 as pkg
    pkg.ShortTermFeatures.PRINT_SPECTROGRAM_SHAPE = False
    return pkg


def long_clip(seed, n, fs):
    """Seeded int16 clip of any length in a few seconds: noise + a slowly varying tone + a level ramp (so that
    frames far apart differ in level, pitch and spectrum), with a DC offset."""
    rng = np.random.default_rng(seed)
    x = rng.normal(0.0, 2500.0, n).astype(np.float32)
    t = np.arange(n, dtype=np.float32)
    f0 = 220.0 + 180.0 * np.sin(2 * np.pi * t / np.float32(7.3 * fs))
    phase = np.cumsum(2 * np.pi * f0 / np.float32(fs), dtype=np.float64).astype(np.float32)
    level = 0.25 + 0.75 * (0.5 + 0.5 * np.sin(2 * np.pi * t / np.float32(31.0 * fs)))
    x = level * (x + 7000.0 * np.sin(phase)) + 37.0
    return np.round(np.clip(x, -32768, 32767)).astype(np.int16)


def test_config3_at_size(P):
    """configs[2]: 44.1 kHz, 60 s, win/step 20/10 ms: feature_extraction (5 999 frames), spectrogram (5 999 rows, the
    last two zero), chromagram (5 998 rows, the last one zero) of one clip; and a batch of 3 through the device API."""
    import torch
    fs, n, w, s = 44100, 2646000, 882, 441
    x = long_clip(3, n, fs)
    F, names = P.ShortTermFeatures.feature_extraction(x, fs, w, s)
    ref, ref_names = O.feature_extraction(x, fs, w, s)
    assert names == ref_names and F.shape == (68, 5999)
    check_features(F, ref, w // 2, "config 3 feature_extraction")
    sp = P.ShortTermFeatures.spectrogram(x, fs, w, s)[0]
    assert sp.shape == (5999, 441) and not sp[5997:].any() and sp[5996].any()
    check_close(sp, O.spectrogram(x, fs, w, s)[0], "config 3 spectrogram", atol=1e-7)
    ch = P.ShortTermFeatures.chromagram(x, fs, w, s)[0]
    assert ch.shape == (5998, 12) and not ch[5997].any()
    check_close(ch, O.chromagram(x, fs, w, s)[0], "config 3 chromagram", atol=1e-6)
    # batched device path at the same size (other clips: shifted copies, so one oracle run covers them)
    clips = np.stack([x, np.roll(x, 12345), x[::-1].copy()])
    out = P.feature_extraction_batch(torch.from_numpy(clips).cuda(), fs, w, s).cpu().numpy()
    check_features(out[0], ref, w // 2, "config 3 batch clip 0")
    check_features(out[2], O.feature_extraction(clips[2], fs, w, s)[0], w // 2, "config 3 batch clip 2")


def test_config4_at_size(P):
    """configs[3]: one hour @16 kHz through mid_feature_extraction, mt 1.0/1.0 s, st 50/25 ms: 143 999 short-term
    frames, 3 600 mid-term windows (57.6 M-sample exact clip sum, ~1 400 work items for one clip)."""
    fs, n = 16000, 57600000
    x = long_clip(4, n, fs)
    mid, st, names = P.MidTermFeatures.mid_feature_extraction(x, fs, 1.0 * fs, 1.0 * fs, 0.050 * fs, 0.025 * fs)
    rm, rs, rn = O.mid_feature_extraction(x, fs, 1.0 * fs, 1.0 * fs, 0.050 * fs, 0.025 * fs)
    assert names == rn and mid.shape == (136, 3600) and st.shape == (68, 143999)
    check_features(st, rs, 400, "config 4 short-term")
    # The pooling itself is held tight against the oracle's pooling of the GPU's own short-term matrix; against the
    # reference's mid-term matrix the short-term tolerance propagates (tests/parity.py: check_mid).
    check_close(mid, O.mid_pool(st, 39, 40), "config 4 pooling of the GPU short-term matrix", rtol=1e-5, atol=1e-6)
    check_mid(mid, rm, rs, "config 4 mid-term")


def test_config5_gathered_two_gpus(P):
    """configs[4] at world_size 2: every rank extracts its shard, NCCL gather to rank 0, rank 0 compares the gathered
    [clips, 68, T] tensor with the oracle clip by clip (tests/dist_gpu_worker.py).  Needs two GPUs."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29631", os.path.join(ROOT, "tests", "dist_gpu_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert res.returncode == 0 and "DIST_GPU_OK" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]
