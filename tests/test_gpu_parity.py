"""GPU parity: the CUDA path (through the C ABI) against reference-generated golden vectors and the oracle."""
import numpy as np
import pytest

from oracle import st_oracle as O
from tests.parity import check_features, check_close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def P():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import pyaudioanalysis_b200 as pkg
    from pyaudioanalysis_b200 import _lib
    assert _lib.lib().b200aa_device_ok() == 0, "not an sm_100 device"
    pkg.ShortTermFeatures.PRINT_SPECTROGRAM_SHAPE = False
    return pkg


# ------------------------------------------------------------------ golden vectors (unmodified reference)
def test_doremi_feature_extraction(P, golden_doremi):
    g = golden_doremi
    F, names = P.ShortTermFeatures.feature_extraction(g["x"], int(g["fs"]), 0.050 * 16000, 0.025 * 16000)
    assert names == list(g["names"])
    assert F.dtype == np.float64 and F.shape == (68, 319)
    check_features(F, g["st"], 400, "doremi 50/25")


def test_doremi_spectrogram_chromagram(P, golden_doremi):
    g = golden_doremi
    sp, t, f = P.ShortTermFeatures.spectrogram(g["x"], 16000, 800, 400)
    assert sp.shape == (319, 400) and not sp[317:].any()
    check_close(sp, g["spectrogram"], "doremi spectrogram", atol=1e-7)
    check_close(np.array(t), g["spec_time"], rtol=1e-12, atol=0); check_close(np.array(f), g["spec_freq"], rtol=1e-12, atol=0)
    ch, t, n = P.ShortTermFeatures.chromagram(g["x"], 16000, 800, 400)
    assert ch.shape == (318, 12) and n == list(g["chroma_names"])
    check_close(ch, g["chromagram"], "doremi chromagram (last row from a clipped frame)", atol=1e-6)
    check_close(np.array(t), g["chroma_time"], rtol=1e-12, atol=0)


def test_doremi_mid(P, golden_doremi):
    g = golden_doremi
    mid, st, names = P.MidTermFeatures.mid_feature_extraction(g["x"], 16000, 16000, 16000, 800, 400)
    assert names == list(g["mid_names"]) and mid.shape == (136, 8) and st.shape == (68, 319)
    check_close(mid, g["mid"], "doremi mid-term")
    check_features(st, g["st"], 400, "doremi st via mid")


def test_reference_pytest_inputs(P, golden_pytests):
    """The reference's own two tests (pytests/test_feature_extraction.py) + values."""
    g = golden_pytests
    F, names = P.ShortTermFeatures.feature_extraction(g["x1"], int(g["fs1"]), 0.050 * 16000, 0.050 * 16000)
    assert F.shape[1] == 20 and F.shape[0] == len(names)
    check_features(F, g["st1"], 400, "1_sec_wav")
    mt, st, mt_names = P.MidTermFeatures.mid_feature_extraction(g["x5"], 16000, 1 * 16000, 1 * 16000, 0.05 * 16000, 0.05 * 16000)
    assert mt.shape[1] == 5 and mt.shape[0] == len(mt_names) == 136
    check_close(mt, g["mid5"], "5_sec_wav mid")
    check_features(st, g["st5"], 400, "5_sec_wav st")


def test_synthetic_goldens(P, golden_synth):
    g = golden_synth
    for idx in (0, 1, 2):
        F, _ = P.ShortTermFeatures.feature_extraction(O.synth_clip(idx, 32000, 16000), 16000, 800, 400)
        check_features(F, g[f"st16_{idx}"], 400, f"synthetic 16k clip {idx}")
    c44 = O.synth_clip(7, 44100, 44100)
    F, _ = P.ShortTermFeatures.feature_extraction(c44, 44100, 882, 441)
    check_features(F, g["st44"], 441, "synthetic 44.1k 20/10 ms")
    check_close(P.ShortTermFeatures.spectrogram(c44, 44100, 882, 441)[0], g["sp44"], "spectrogram 44.1k", atol=1e-7)
    check_close(P.ShortTermFeatures.chromagram(c44, 44100, 882, 441)[0], g["ch44"], "chromagram 44.1k", atol=1e-6)


def test_float_input_odd_window(P, golden_synth):
    cf = O.synth_clip(11, 20000, 22050).astype(np.float64) * 0.37 + 11.5
    F, names = P.ShortTermFeatures.feature_extraction(cf, 22050, 551, 200, deltas=False)
    assert len(names) == 34
    check_features(F, golden_synth["st_float_551"], 275, "float64 input, window 551, step 200, no deltas")


def test_other_sample_formats(P):
    """Integer formats other than int16: 8-bit and unsigned 16-bit PCM are exact in the device formats; 32-bit PCM (as
    scipy returns 24 / 32-bit WAV files) goes through float32 -- the path is scale invariant and the 2^-24 relative
    rounding of a sample is far below the tolerance."""
    rng = np.random.default_rng(17)
    base = O.synth_clip(91, 24000, 16000)
    x32 = base.astype(np.int32) * 65536 + rng.integers(-30000, 30000, base.shape[0])          # 32-bit PCM with live low bits
    x24 = (base.astype(np.int32) * 256 + rng.integers(-100, 100, base.shape[0])).astype(np.int32)
    u8 = ((base // 256) + 128).astype(np.uint8)
    u16 = (base.astype(np.int32) + 32768).astype(np.uint16)
    for name, x in (("int32", x32), ("24-bit in int32", x24), ("uint8", u8), ("uint16", u16), ("float64", base.astype(np.float64) / 32768.0)):
        F, _ = P.ShortTermFeatures.feature_extraction(x, 16000, 800, 400)
        check_features(F, O.feature_extraction(x, 16000, 800, 400)[0], 400, "input format " + name)


def test_one_second_windows(P, golden_synth):
    """music_thumbnailing calls the path with 1 s windows (audioSegmentation.py:1137-1139)."""
    F, _ = P.ShortTermFeatures.feature_extraction(O.synth_clip(13, 80000, 16000), 16000, 16000, 16000)
    check_features(F, golden_synth["st_win16000"], 8000, "window = step = 16000")


def test_large_windows(P):
    """Windows whose transform does not fit shared memory run through the global-memory form of the generic kernel:
    1 s windows at 44.1 / 22.05 kHz (music_thumbnailing, audioSegmentation.py:1137-1139) and 30 000 / 15 000 samples,
    against golden values of the unmodified reference (tests/golden/bigwin.npz, oracle/make_golden_r2.py)."""
    from tests.conftest import load_golden
    g = load_golden("bigwin.npz")
    for fs in (44100, 22050):
        F, _ = P.ShortTermFeatures.feature_extraction(g["x_%d" % fs], fs, fs, fs)
        check_features(F, g["st_%d" % fs], fs // 2, "window = step = %d" % fs)
    F, _ = P.ShortTermFeatures.feature_extraction(g["x_30000"], 32000, 30000, 15000)
    check_features(F, g["st_30000"], 15000, "window 30000 step 15000")
    x = g["x_44100"]
    sp = P.ShortTermFeatures.spectrogram(x, 44100, 44100, 22050)[0]
    check_close(sp, O.spectrogram(x, 44100, 44100, 22050)[0], "spectrogram window 44100", atol=1e-7)
    # 2^17-sample window (above any use the reference makes of the path) still works
    xl = O.synth_clip(77, 3 * 131072 + 5, 48000)
    F, _ = P.ShortTermFeatures.feature_extraction(xl, 48000, 131072, 131072)
    check_features(F, O.feature_extraction(xl, 48000, 131072, 131072)[0], 65536, "window 2^17")


def test_mid_awkward_ratio(P, golden_synth):
    mid, st, _ = P.MidTermFeatures.mid_feature_extraction(O.synth_clip(3, 50000, 16000), 16000, 16000, 8000, 800, 400)
    check_close(mid, golden_synth["mid_16000_8000"], "mid 1.0/0.5 s")


@pytest.mark.parametrize("fs,w,s,n,exc,text", [
    (4000, 100, 50, 50, IndexError, None),             # mel bank fails before the (empty) frame loop
    (4000, 100, 50, 1000, IndexError, None),
    (4000, 400, 200, 100, IndexError, None),
    (8000, 160, 80, 100, ValueError, "need at least one array"),   # no frames: the chroma scatter is never reached
    (8000, 160, 80, 1000, ValueError, "chroma"),
])
def test_error_precedence(P, fs, w, s, n, exc, text):
    """Exception types of the unmodified reference on these inputs (tests/test_oracle_vs_reference.py checks
    the oracle against the reference's stored values)."""
    x = O.synth_clip(1, n, fs)
    for fn in (lambda: P.ShortTermFeatures.feature_extraction(x, fs, w, s),
               lambda: P.MidTermFeatures.mid_feature_extraction(x, fs, 4 * w, 4 * w, w, s)):
        with pytest.raises(exc) as e:
            fn()
        if text:
            assert text in str(e.value)
        with pytest.raises(exc):
            O.feature_extraction(x, fs, w, s)


def test_edges(P, golden_edges):
    g = golden_edges
    S = P.ShortTermFeatures
    Fz, _ = S.feature_extraction(np.zeros(4000, dtype=np.int16), 16000, 800, 400)
    check_features(Fz, g["zeros"], 400, "all-zero clip")
    assert abs(Fz[8, 0] - (-99.00180475419432)) < 1e-3
    Fk, _ = S.feature_extraction(np.full(4000, 1234, dtype=np.int16), 16000, 800, 400)
    check_features(Fk[:8], g["const"][:8], 400, "constant clip (time/spectral rows)")
    for n in (800, 1199, 1200):
        F, _ = S.feature_extraction(O.synth_clip(5, n, 16000), 16000, 800, 400)
        check_features(F, g[f"n{n}"], 400, f"N={n}")
    with pytest.raises(ValueError, match="need at least one array"):
        S.feature_extraction(O.synth_clip(5, 799, 16000), 16000, 800, 400)
    with pytest.raises(ValueError):
        S.feature_extraction(O.synth_clip(5, 4000, 8000), 8000, 160, 80)     # chroma else-branch of the reference
    Fs, _ = S.feature_extraction(g["silence_x"], 16000, 800, 400)
    # Frames 8..15 are digital silence: the reference's non-DC bins there are float64 round-off
    # (~1e-19) passed through log10(. + eps), which makes its mfcc_2..13 = 3.1e-5 -- noise that even
    # the float64 oracle does not reproduce (it differs by 3.6e-5, tests/test_oracle_golden.py).  The
    # GPU transforms (x - x[0]) and gets exact zeros there.  Those frames (and the deltas that touch
    # them) are held to atol 1e-4 instead of 1e-5; everything else to the standard tolerance.
    noisy = np.zeros(Fs.shape[1], bool); noisy[8:17] = True
    check_features(Fs[:, ~noisy], g["silence"][:, ~noisy], 400, "digital silence inside a clip with DC offset")
    check_close(Fs[:, noisy], g["silence"][:, noisy], "digitally silent frames", rtol=1e-4, atol=1e-4)
    cc = O.synth_clip(22, 16300, 16000)
    check_close(S.chromagram(cc, 16000, 800, 400)[0], g["chroma_clipped"], "chromagram, clipped last frame", atol=1e-6)
    check_close(S.spectrogram(cc, 16000, 800, 400)[0], g["spec_16300"], "spectrogram N=16300", atol=1e-7)


# ------------------------------------------------------------------ oracle on seeded inputs
@pytest.mark.parametrize("fs,w,s,n", [(16000, 800, 400, 48000), (16000, 800, 800, 16000), (16000, 640, 160, 20000),
                                      (44100, 882, 441, 30000), (8000, 400, 200, 12000), (22050, 1102, 551, 30000),
                                      (48000, 2400, 1200, 60000), (16000, 1024, 512, 20000), (16000, 883, 300, 9000),
                                      (16000, 400, 160, 20000), (16000, 480, 160, 20000), (8000, 600, 300, 12000),
                                      (16000, 400, 133, 9000), (16000, 480, 480, 9600), (16000, 320, 160, 12000),
                                      (16000, 640, 321, 12000), (8000, 320, 80, 8000)])
def test_oracle_configs(P, fs, w, s, n):
    x = O.synth_clip(100 + w, n, fs)
    ref, names = O.feature_extraction(x, fs, w, s)
    F, names2 = P.ShortTermFeatures.feature_extraction(x, fs, w, s)
    assert names == names2
    check_features(F, ref, w // 2, f"fs={fs} w={w} s={s}")


def test_batch_and_ragged(P):
    import torch
    clips = np.stack([O.synth_clip(i, 32000, 16000) for i in range(5)])
    d = torch.from_numpy(clips).cuda()
    out = P.feature_extraction_batch(d, 16000, 800, 400)
    assert out.shape == (5, 68, 79) and out.dtype == torch.float32 and out.is_cuda
    for i in range(5):
        check_features(out[i].cpu().numpy(), O.feature_extraction(clips[i], 16000, 800, 400)[0], 400, f"batch clip {i}")
    # the work split (frames per CTA run, halo recomputation) depends on the batch size; results must not
    alone = P.feature_extraction_batch(d[2:3], 16000, 800, 400)
    assert torch.equal(alone[0], out[2]), "result depends on how the batch was split across CTAs"
    lens = torch.tensor([32000, 800, 12345, 31999, 20000], dtype=torch.int64, device="cuda")
    out = P.feature_extraction_batch(d, 16000, 800, 400, lengths=lens)
    for i, L in enumerate(lens.tolist()):
        ref = O.feature_extraction(clips[i][:L], 16000, 800, 400)[0]
        got = out[i].cpu().numpy()
        check_features(got[:, :ref.shape[1]], ref, 400, f"ragged clip {i}")
        assert not got[:, ref.shape[1]:].any()
    f32 = torch.from_numpy(clips.astype(np.float32) * 3.0).cuda()
    outf = P.feature_extraction_batch(f32, 16000, 800, 400, deltas=False)
    for i in range(5):
        check_features(outf[i].cpu().numpy(), O.feature_extraction(clips[i], 16000, 800, 400, deltas=False)[0], 400, f"f32 clip {i}")


def test_work_stealing_is_invisible(P, monkeypatch):
    """More pair steps than resident warps, ragged lengths, and the steal-half scheduler (csrc/sched.cuh) forced to hand
    ranges over all the time (claims of one pair, any remainder stolen): outputs are bit-identical to the default
    settings' and to a clip processed alone -- results do not depend on which warp computed which pairs -- for the pair
    kernel (800 / 400) and the solo kernel (882 / 441)."""
    import torch
    rng = np.random.default_rng(77)
    base = np.stack([O.synth_clip(200 + i, 48000, 16000) for i in range(8)])
    clips = torch.from_numpy(np.concatenate([np.roll(base, 37 * k, axis=1) for k in range(40)])).cuda()       # 320 clips x 3 s
    lens = torch.from_numpy(rng.integers(700, 48001, size=clips.shape[0]).astype(np.int64)).cuda()
    lens[:8] = 48000
    for fs, w, s in ((16000, 800, 400), (44100, 882, 441)):
        monkeypatch.delenv("B200AA_PAIR_STEAL", raising=False)
        ref = P.feature_extraction_batch(clips, fs, w, s, lengths=lens).clone()
        for setting in ("1,2", "3,7", "64,2"):
            monkeypatch.setenv("B200AA_PAIR_STEAL", setting)
            got = P.feature_extraction_batch(clips, fs, w, s, lengths=lens)
            assert torch.equal(got, ref), "results depend on the work distribution (%s, window %d)" % (setting, w)
        monkeypatch.delenv("B200AA_PAIR_STEAL", raising=False)
        alone = P.feature_extraction_batch(clips[5:6], fs, w, s)
        assert torch.equal(alone[0], ref[5])
        for i in (0, 3):
            check_features(ref[i].cpu().numpy(), O.feature_extraction(base[i], fs, w, s)[0], w // 2, "stolen clip %d window %d" % (i, w))


def test_directory_feature_extraction(P, tmp_path):
    """SURVEY 8f rank 1: long-term averaged mid-term vectors per file of a folder, against the reference's own output
    on its 3_class test clips (8 kHz, 1 s, 12 per class; the silence class exercises near-digital-silence audio)."""
    from scipy.io import wavfile
    from tests.conftest import load_golden
    g = load_golden("dirs.npz")
    P.MidTermFeatures.VERBOSE = False
    dirs = []
    for cls in ("music", "silence", "speech"):
        d = tmp_path / cls
        d.mkdir()
        for name, x in zip(g[cls + "_files"], g[cls + "_x"]):
            wavfile.write(str(d / str(name)), int(g["fs"]), x)
        dirs.append(str(d))
        feats, files, names = P.MidTermFeatures.directory_feature_extraction(str(d), 1.0, 1.0, 0.05, 0.05, compute_beat=False)
        assert names == list(g["names"]) and [f.split("/")[-1] for f in files] == list(g[cls + "_files"])
        assert feats.shape == (12, 136)
        check_close(feats, g[cls + "_feats"], f"directory_feature_extraction {cls}", rtol=2e-4, atol=2e-5)
    f3, classes, fn3 = P.MidTermFeatures.multiple_directory_feature_extraction(dirs, 1.0, 1.0, 0.05, 0.05)
    assert classes == ["music", "silence", "speech"] and len(f3) == 3 and f3[0].shape == (12, 136)
    # compute_beat (the default): bpm / ratio of this package's own beat_extraction (reference MidTermFeatures.py:18-84)
    # on the GPU short-term rows.  Peak picking is discrete, so the expectation is built from the float64 oracle's rows
    # and compared per file: the tempo bin must agree on (nearly) every file.
    fb, _, nb = P.MidTermFeatures.directory_feature_extraction(dirs[0], 1.0, 1.0, 0.05, 0.05)
    assert fb.shape == (12, 138) and nb == list(g["names"]) + ["bpm", "ratio"]
    check_close(fb[:, :136], g["music_feats"], "directory_feature_extraction with beat", rtol=2e-4, atol=2e-5)
    exp = [P.MidTermFeatures.beat_extraction(O.feature_extraction(x, int(g["fs"]), 400, 400)[0], 0.05) for x in g["music_x"]]
    same = sum(1 for k in range(12) if abs(fb[k, 136] - exp[k][0]) < 1e-9 and abs(fb[k, 137] - exp[k][1]) < 1e-6)
    assert same >= 11, (same, fb[:, 136:], exp)
    one = tmp_path / "one"
    one.mkdir()
    wavfile.write(str(one / "a.wav"), int(g["fs"]), g["music_x"][0])
    f1, _, _ = P.MidTermFeatures.directory_feature_extraction(str(one), 1.0, 1.0, 0.05, 0.05, compute_beat=False)
    assert f1.shape == (136,)                       # the reference returns a 1-D vector for a single file
    empty = tmp_path / "none"
    empty.mkdir()
    f0, l0, _ = P.MidTermFeatures.directory_feature_extraction(str(empty), 1.0, 1.0, 0.05, 0.05, compute_beat=False)
    assert f0.shape == (0,) and l0 == []


def test_file_wrappers(P, tmp_path):
    """SURVEY 8f rank 1/3: no-averaging directory wrapper and the .npy / CSV writers (MidTermFeatures.py:263-377)."""
    from scipy.io import wavfile
    P.MidTermFeatures.VERBOSE = False
    clips = [O.synth_clip(300 + i, n, 16000) for i, n in enumerate((40000, 24000, 40000))]
    stereo = np.stack([clips[1], clips[1][::-1]], axis=1)            # a 2-channel file: (L/2)+(R/2)
    d = tmp_path / "wavs"
    d.mkdir()
    wavfile.write(str(d / "a.wav"), 16000, clips[0])
    wavfile.write(str(d / "b.wav"), 16000, stereo)
    wavfile.write(str(d / "c.wav"), 16000, clips[2])
    from pyaudioanalysis_b200 import audioio
    pb = audioio.PinnedBatch(2, 40000)                     # page-locked staging: mono PCM16 files are read straight into it
    pb.fill(0, str(d / "a.wav"))
    pb.fill(1, str(d / "c.wav"))
    assert pb.direct == 2 and (pb.array[0] == clips[0]).all() and (pb.array[1] == clips[2]).all()
    X, idx, files = P.MidTermFeatures.directory_feature_extraction_no_avg(str(d), 1.0, 0.5, 0.05, 0.025)
    mono_b = (stereo[:, 1] / 2) + (stereo[:, 0] / 2)
    refs = [O.mid_feature_extraction(c, 16000, 16000, 8000, 800, 400)[0] for c in (clips[0], mono_b, clips[2])]
    assert X.shape == (sum(r.shape[1] for r in refs), 136) and len(files) == 3
    check_close(X, np.vstack([r.T for r in refs]), "directory_feature_extraction_no_avg", rtol=2e-4, atol=2e-5)
    assert list(idx[:refs[0].shape[1]]) == [0.0] * refs[0].shape[1] and idx[-1] == 2.0
    out = str(tmp_path / "feat")
    P.MidTermFeatures.mid_feature_extraction_to_file(str(d / "a.wav"), 1.0, 1.0, 0.05, 0.05, out, store_short_features=True, store_csv=True)
    mt, st = np.load(out + "_mt.npy"), np.load(out + "_st.npy")
    rm, rs, _ = O.mid_feature_extraction(clips[0], 16000, 16000, 16000, 800, 800)
    assert mt.dtype == np.float64 and mt.shape == rm.shape and st.shape == rs.shape
    check_close(mt, rm, "_mt.npy", rtol=2e-4, atol=2e-5)
    csv = np.loadtxt(out + "_mt.csv", delimiter=",")
    assert csv.shape == mt.T.shape
    np.testing.assert_allclose(csv, mt.T, rtol=1e-12)
    P.MidTermFeatures.mid_feature_extraction_file_dir(str(d), 1.0, 1.0, 0.05, 0.05)
    assert (d / "c.wav_mt.npy").exists()


def test_host_pipeline(P):
    """Pinned-host batch API = one call of the C ABI's b200aa_st_features_host (chunked copies + kernels on three
    streams inside the library for big batches, single stream for small ones) equals the device-resident path."""
    import torch
    from pyaudioanalysis_b200.hostpipe import HostPipeline
    clips = np.stack([O.synth_clip(200 + i, 16000, 16000) for i in range(7)])
    pipe = HostPipeline(16000, 800, 400, 16000, max_clips=7, device=0)
    pipe.h_in[:] = clips
    got = pipe.run().copy()
    ref = P.feature_extraction_batch(torch.from_numpy(clips).cuda(), 16000, 800, 400).cpu().numpy()
    assert (got == ref).all()
    again = pipe.run(clips[:4])                       # pageable input works too
    assert (again == ref[:4]).all()
    with pytest.raises(TypeError):
        pipe.run(clips.astype(np.float32))            # no silent dtype conversion
    with pytest.raises(ValueError):
        pipe.run(clips[:, :8000])
    # a batch large enough for the chunked three-stream form (> 2 chunks of ~32 MB): 250 clips of 10 s
    big = np.stack([O.synth_clip(900 + (i % 5), 160000, 16000) for i in range(250)])
    big[5:] = np.roll(big[5:], 7, axis=1)
    pipe2 = HostPipeline(16000, 800, 400, 160000, max_clips=250, device=0)
    pipe2.h_in[:] = big
    got2 = pipe2.run()
    ref2 = P.feature_extraction_batch(torch.from_numpy(big).cuda(), 16000, 800, 400).cpu().numpy()
    assert (got2 == ref2).all()
    check_features(got2[3], O.feature_extraction(big[3], 16000, 800, 400)[0], 400, "chunked host pipeline clip 3")


def test_kernel_kinds_agree(P):
    """Every kernel that exists for a window (2 = warp-autonomous pair kernel, 3 = warp-autonomous per-frame ("solo") kernel,
    1 = register-tiled CTA kernel, 0 = generic) must agree with the oracle; the default plan picks the fastest one."""
    import torch
    from pyaudioanalysis_b200._lib import Plan
    for fs, w, s in [(16000, 800, 400), (44100, 882, 441), (16000, 800, 800), (16000, 800, 200), (8000, 400, 200),
                     (16000, 400, 160), (16000, 480, 240), (8000, 600, 300), (16000, 640, 320), (16000, 320, 160),
                     (16000, 1024, 512), (16000, 512, 256), (16000, 512, 128), (48000, 960, 480), (16000, 1024, 300),
                     (16000, 800, 333), (44100, 882, 882), (44100, 882, 300), (16000, 400, 400), (8000, 600, 150)]:
        clips = np.stack([O.synth_clip(40 + i, 24000 + 7 * i, fs)[:24000] for i in range(3)])
        d = torch.from_numpy(clips).cuda()
        refs = [O.feature_extraction(clips[i], fs, w, s)[0] for i in range(3)]
        kinds = set()
        for prefer in (-1, 2, 3, 1, 0):
            pl = Plan(fs, w, s).prefer_kernel(prefer)
            kind = pl.kernel_kind()
            if prefer >= 0 and kind != prefer:
                continue                        # that kernel does not exist for this window
            kinds.add(kind)
            got = P.feature_extraction_batch(d, fs, w, s, plan=pl).cpu().numpy()
            for i in range(3):
                check_features(got[i], refs[i], w // 2, f"kernel kind {kind} (prefer {prefer}) fs={fs} w={w} s={s}")
        assert 0 in kinds
        if w in (320, 480, 512, 640, 800, 960, 1024):
            assert 2 in kinds and Plan(fs, w, s).kernel_kind() == 2
        if w in (882, 400, 600):
            assert 3 in kinds and 1 in kinds and Plan(fs, w, s).kernel_kind() == 3
        pg = Plan(fs, w, s)
        pg.force_generic(True)
        assert pg.kernel_kind() == 0


def test_row_kernels_agree(P):
    """spectrogram / chromagram through the default kernel (solo for 882 / 400 / 600, CTA for 800 / 320 / 480 / 640,
    generic for the pair-only windows 512 / 960 / 1024), the CTA kernel where the window has one, the generic kernel,
    and the oracle."""
    import torch
    from pyaudioanalysis_b200._lib import Plan
    for fs, w, s, n in [(16000, 800, 400, 40000), (44100, 882, 441, 50000), (16000, 800, 800, 24000), (16000, 800, 200, 16400),
                        (16000, 400, 160, 16000), (8000, 600, 300, 12000), (44100, 882, 882, 30000), (44100, 882, 300, 20001),
                        (16000, 320, 160, 12000), (16000, 480, 240, 12000), (16000, 640, 320, 16000),
                        (16000, 512, 256, 16000), (48000, 960, 480, 48000), (16000, 1024, 512, 16000)]:
        clips = np.stack([O.synth_clip(60 + i, n, fs) for i in range(3)])
        d = torch.from_numpy(clips).cuda()
        plans = [Plan(fs, w, s), Plan(fs, w, s).prefer_kernel(1), Plan(fs, w, s)]
        plans[2].force_generic(True)
        for fn, ofn, atol in ((P.spectrogram_batch, O.spectrogram, 1e-7), (P.chromagram_batch, O.chromagram, 1e-6)):
            refs = [ofn(clips[i], fs, w, s)[0] for i in range(3)]
            for pl, what in zip(plans, ("default", "CTA", "generic")):
                a = fn(d, fs, w, s, plan=pl).cpu().numpy()
                for i in range(3):
                    check_close(a[i], refs[i], f"{fn.__name__} {what} plan (kind {pl.kernel_kind()}) fs={fs} w={w} s={s}", atol=atol)
    # a clipped last frame shorter than num_fft makes the reference's scatter raise ValueError (:288)
    bad = O.synth_clip(60, 16300, 16000)
    with pytest.raises(ValueError):
        O.chromagram(bad, 16000, 800, 200)
    with pytest.raises(ValueError):
        P.ShortTermFeatures.chromagram(bad, 16000, 800, 200)


# ------------------------------------------------------------------ full-size properties (BASELINE configs[1])
def test_full_size_properties(P):
    """1000 x 10 s @16 kHz: no oracle at this size -- use properties that do not depend on it."""
    import torch
    torch.manual_seed(0)
    B, N = 1000, 160000
    base = (3000.0 * torch.randn(B, N, device="cuda")).round().clamp(-16000, 16000).to(torch.int16)
    base[1] = base[0]                      # identical clips -> identical features
    base[3] = (base[2].to(torch.int32) * 2).to(torch.int16)   # gain 2 (no clipping): normalisation removes it
    out = P.feature_extraction_batch(base, 16000, 800, 400)
    assert out.shape == (B, 68, 399) and torch.isfinite(out).all()
    assert torch.equal(out[0], out[1])
    torch.testing.assert_close(out[3], out[2], rtol=1e-4, atol=2e-5)
    # deltas are the first difference of the base rows, zero in column 0
    torch.testing.assert_close(out[:, 34:, 1:], out[:, :34, 1:] - out[:, :34, :-1], rtol=0, atol=0)
    assert not out[:, 34:, 0].any()
    # spot-check five clips against the oracle
    for i in (0, 2, 499, 998, 999):
        check_features(out[i].cpu().numpy(), O.feature_extraction(base[i].cpu().numpy(), 16000, 800, 400)[0], 400, f"cfg2 clip {i}")
    # chroma rows sum to <= 1 and are non-negative; energy equals mean square of normalised samples
    assert (out[:, 21:33] >= 0).all()
