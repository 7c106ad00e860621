"""CPU: host-side pieces next to the GPU path (SURVEY 8f ranks 2 and 4): beat_extraction / peak picking against golden
values of the unmodified reference, and the file decoders (WAV layout walk, direct-into-buffer decode, AIFF, stereo)."""
import os
import struct
import wave

import numpy as np
import pytest

from tests.conftest import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


BEAT_ROWS = 19          # beat_extraction reads short-term rows 0-18 only (reference MidTermFeatures.py:31-32)


def beat_walks():
    """Random-walk feature matrices 4-7 of tests/golden/beat.npz, regenerated from their seed."""
    rng = np.random.default_rng(9)
    return [np.cumsum(rng.standard_normal((68, 300 + 40 * i)), axis=1) * 0.05 + rng.standard_normal((68, 1)) for i in range(4, 8)]


def peak_inputs():
    """Seeded (signal, peakdet threshold, feature matrix) triples of test_beat_extraction_against_imported_reference."""
    rng = np.random.default_rng(3)
    out = []
    for k in range(6):
        v = np.cumsum(rng.standard_normal(400)) * (0.1 + k)
        delta = 2.0 * np.abs(np.diff(v)).mean()
        out.append((v, delta, np.cumsum(rng.standard_normal((34, 200 + 30 * k)), axis=1)))
    return out


def test_beat_extraction_matches_reference_golden():
    """tests/golden/beat.npz: MidTermFeatures.beat_extraction of the unmodified reference (oracle/make_golden_r2.py;
    numpy.Inf / numpy.NaN aliased for NumPy 2) on 8 feature matrices: the short-term features of four pulse clips (rows
    0-18 stored, the others zero) and four seeded random walks."""
    from pyaudioanalysis_b200.MidTermFeatures import beat_extraction
    g = load_golden("beat.npz")
    walks = beat_walks()
    for i in range(int(g["n"])):
        if i < 4:
            st = np.zeros((68, g["st_%d" % i].shape[1]))
            st[:BEAT_ROWS] = g["st_%d" % i]
        else:
            st = walks[i - 4]
            assert st.sum() == pytest.approx(float(g["sum_%d" % i]), rel=1e-12), "random walk %d is not the golden input" % i
        bpm, ratio = beat_extraction(st, float(g["win_%d" % i]))
        assert bpm == pytest.approx(float(g["bpm_%d" % i]), rel=1e-12), i
        assert ratio == pytest.approx(float(g["ratio_%d" % i]), rel=1e-12, abs=1e-15), i


def test_beat_extraction_against_imported_reference():
    """Peak picking and beat_extraction against the reference's utilities.peakdet / MidTermFeatures.beat_extraction on
    seeded inputs (values in tests/golden/beat.npz, oracle/make_golden_r2.py)."""
    from pyaudioanalysis_b200.MidTermFeatures import beat_extraction, _peak_positions
    g = load_golden("beat.npz")
    for k, (v, delta, st) in enumerate(peak_inputs()):
        assert _peak_positions(v, delta) == g["peaks_%d" % k].tolist()
        for win, ref in zip((0.05, 0.025, 0.1), g["beats_%d" % k]):
            assert beat_extraction(st, win) == pytest.approx(tuple(ref), rel=1e-12)
    flat = np.ones((34, 100))
    assert beat_extraction(flat, 0.05) == pytest.approx(tuple(g["beats_flat"]))


def _write_wav(path, data, fs, extra_chunk=False):
    with wave.open(path, "wb") as w:
        w.setnchannels(1 if data.ndim == 1 else data.shape[1])
        w.setsampwidth(2)
        w.setframerate(fs)
        w.writeframes(np.ascontiguousarray(data).astype("<i2").tobytes())
    if extra_chunk:          # a LIST chunk in front of the data chunk
        raw = open(path, "rb").read()
        i = raw.index(b"data")
        lst = b"LIST" + struct.pack("<I", 5) + b"abcde\x00"
        out = raw[:i] + lst + raw[i:]
        out = out[:4] + struct.pack("<I", len(out) - 8) + out[8:]
        open(path, "wb").write(out)


def test_wav_layout_and_direct_decode(tmp_path):
    from scipy.io import wavfile
    from pyaudioanalysis_b200 import audioio
    rng = np.random.default_rng(1)
    x = rng.integers(-30000, 30000, 12345).astype(np.int16)
    p = str(tmp_path / "a.wav")
    _write_wav(p, x, 16000)
    assert audioio.wav_pcm16_layout(p)[:3] == (16000, 1, 12345)
    dst = np.zeros(12345, np.int16)
    assert audioio.read_wav_into(p, dst) == 16000 and (dst == x).all()
    assert audioio.read_wav_into(p, np.zeros(12000, np.int16)) is None          # wrong length: caller falls back
    p2 = str(tmp_path / "b.wav")
    _write_wav(p2, x, 8000, extra_chunk=True)
    assert audioio.wav_pcm16_layout(p2)[:3] == (8000, 1, 12345)
    dst[:] = 0
    assert audioio.read_wav_into(p2, dst) == 8000 and (dst == x).all()
    fs, y = audioio.read_audio_file(p2)
    assert fs == 8000 and (y == x).all()
    st = np.stack([x, x[::-1]], axis=1)
    p3 = str(tmp_path / "c.wav")
    _write_wav(p3, st, 22050)
    assert audioio.wav_pcm16_layout(p3)[:3] == (22050, 2, 12345)
    assert audioio.read_wav_into(p3, dst) is None                                 # stereo is decoded + mixed on the host
    fs, y = audioio.read_audio_file(p3)
    mono = audioio.stereo_to_mono(y)
    np.testing.assert_array_equal(mono, (st[:, 1] / 2) + (st[:, 0] / 2))          # audioBasicIO.py:166
    p4 = str(tmp_path / "f.wav")
    wavfile.write(p4, 16000, (x / 32768.0).astype(np.float32))                    # float WAV: not PCM16 -> scipy path
    assert audioio.wav_pcm16_layout(p4) is None
    assert audioio.read_audio_file(p4)[1].dtype == np.float32
    assert audioio.wav_pcm16_layout(str(tmp_path / "missing.wav")) is None


def test_aiff_and_unknown_formats(tmp_path):
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import aifc
    from pyaudioanalysis_b200 import audioio
    x = (np.arange(5000) * 7 % 20000 - 10000).astype(np.int16)
    p = str(tmp_path / "t.aiff")
    with aifc.open(p, "wb") as a:
        a.setnchannels(1)
        a.setsampwidth(2)
        a.setframerate(11025)
        a.writeframes(x.astype(">i2").tobytes())
    fs, y = audioio.read_audio_file(p)
    assert fs == 11025 and y.dtype == np.int16 and (y == x).all()
    with pytest.raises(audioio.DecodeError):
        audioio.read_audio_file(str(tmp_path / "x.flac"))
    open(str(tmp_path / "bad.aif"), "wb").write(b"not an aiff file")
    with pytest.raises(audioio.DecodeError):
        audioio.read_audio_file(str(tmp_path / "bad.aif"))
    try:
        import pydub  # noqa: F401
    except Exception:
        open(str(tmp_path / "s.mp3"), "wb").write(b"\\x00" * 64)
        with pytest.raises(audioio.DecodeError):
            audioio.read_audio_file(str(tmp_path / "s.mp3"))


def test_numa_helpers():
    from pyaudioanalysis_b200 import numa
    assert numa.parse_cpulist("0-3,8,10-11") == [0, 1, 2, 3, 8, 10, 11]
    assert numa.parse_cpulist("") == []
    assert numa.bind_to_gpu(0) is None or "node" in numa.bind_to_gpu(0)       # no GPU here: no change, no exception
