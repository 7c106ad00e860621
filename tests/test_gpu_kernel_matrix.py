"""Every short-term kernel against the float64 oracle, across the inputs that pick its code paths.

Which kernel runs, and which path inside it, depends on the window (kernel table below), the hop (the pair kernel's
shared half frames at step == window / 2; the CTA kernel's 8-sample runs, even and odd hops), the dtype, the clip stride
and the base address (16-byte vector loads, TMA staging), the ``lengths`` vector (ragged clips, clips without a
frame) and the clip's statistics (ties with the mean in the zero-crossing count, the sign of the larger excursion,
quiet float clips).  Each test below runs every kernel that serves a window and compares each with the oracle at the
standard tolerance of ``tests/parity.py``.

Samples past a clip's length and the gaps between padded clips hold loud full-scale noise, so a kernel that reads
past a clip's end changes its features; output buffers are pre-filled with a NaN payload, so a column a kernel should
leave alone, or one it never writes, shows up bit for bit.
"""
import numpy as np
import pytest

from oracle import st_oracle as O
from tests.parity import check_features, check_close

pytestmark = pytest.mark.gpu

# ---------------------------------------------------------------------------------------------- kernel table
PAIR, SOLO, CTA, GENERIC = 2, 3, 1, 0
KIND_NAME = {PAIR: "pair", SOLO: "solo", CTA: "CTA", GENERIC: "generic"}
KERNEL_WINDOWS = {
    PAIR: frozenset({320, 480, 512, 640, 800, 960, 1024}),
    SOLO: frozenset({400, 600, 882}),
    CTA: frozenset({320, 400, 480, 600, 640, 800, 882}),
}                                                    # the generic kernel serves every window


def feature_kernels(w):
    """Kernels of the feature path for window w, in the order the default plan prefers them."""
    return [k for k in (PAIR, SOLO, CTA) if w in KERNEL_WINDOWS[k]] + [GENERIC]


def row_kernels(w):
    """Spectrogram / chromagram rows: the pair kernel has no row mode (its windows go to the CTA or generic kernel)."""
    return [k for k in (SOLO, CTA) if w in KERNEL_WINDOWS[k]] + [GENERIC]


NAN_BITS = np.uint32(0x7FC0DEAD)                     # a quiet NaN no arithmetic produces


def nan_filled(shape):
    import torch
    t = torch.empty(shape, dtype=torch.float32, device="cuda")
    t.view(torch.int32).fill_(int(NAN_BITS))
    return t


@pytest.fixture(scope="module")
def P():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import pyaudioanalysis_b200 as pkg
    from pyaudioanalysis_b200 import _lib
    assert _lib.lib().b200aa_device_ok() == 0, "not an sm_100 device"
    return pkg


@pytest.fixture(scope="module")
def plans(P):
    """plans(fs, w, s, kind) -> a cached plan restricted to that kernel (asserted)."""
    from pyaudioanalysis_b200._lib import Plan
    cache = {}

    def get(fs, w, s, kind):
        key = (fs, w, s, kind)
        if key not in cache:
            pl = Plan(fs, w, s).prefer_kernel(kind)
            assert pl.kernel_kind() == kind, (key, pl.kernel_kind())
            cache[key] = pl
        return cache[key]
    return get


def test_kernel_table(P):
    from pyaudioanalysis_b200._lib import Plan
    fs_of = {882: 44100, 551: 22050, 1102: 22050, 960: 48000, 2400: 48000}
    for w in sorted(set().union(*KERNEL_WINDOWS.values()) | {551, 1102, 2400}):
        fs = fs_of.get(w, 16000)
        for kind in (PAIR, SOLO, CTA, GENERIC):
            served = kind == GENERIC or w in KERNEL_WINDOWS[kind]
            got = Plan(fs, w, w // 2).prefer_kernel(kind).kernel_kind()
            assert got == (kind if served else GENERIC), "window %d, prefer %s: kernel kind %d" % (w, KIND_NAME[kind], got)
        assert Plan(fs, w, w // 2).kernel_kind() == feature_kernels(w)[0], "default kernel of window %d" % w
        pg = Plan(fs, w, w // 2)
        pg.force_generic(True)
        assert pg.kernel_kind() == GENERIC


# ---------------------------------------------------------------------------------------------- inputs
GAIN, OFFSET = 0.7071, 123.25                         # float32 clips: int16 clip * GAIN + OFFSET

# (extra columns of the backing tensor, first column of the view): padded = stride N + 8 with an aligned base;
# misaligned = odd stride, base one sample off; shifted = stride a multiple of 8 samples, base one sample off
LAYOUTS = {"contiguous": (0, 0), "padded": (8, 0), "misaligned": (3, 1), "shifted": (8, 1)}


def as_dtype(x16, dtype):
    if dtype == "int16":
        return x16
    return (x16.astype(np.float64) * GAIN + OFFSET).astype(np.float32)


def loud_noise(rng, shape, dtype):
    if dtype == "int16":
        return rng.integers(-32768, 32768, size=shape).astype(np.int16)
    return (rng.uniform(-1.0, 1.0, size=shape) * 32768.0 * GAIN * 4 + OFFSET).astype(np.float32)


def device_clips(clips, lengths, layout, seed=0):
    """CUDA [B, N] view in the given layout; samples past each clip's length and the gaps hold loud noise."""
    import torch
    B, N = clips.shape
    extra, first = LAYOUTS[layout]
    big = loud_noise(np.random.default_rng(seed), (B, N + extra), "int16" if clips.dtype == np.int16 else "float32")
    for i in range(B):
        L = N if lengths is None else lengths[i]
        big[i, first:first + L] = clips[i, :L]
    view = torch.from_numpy(big).cuda()[:, first:first + N]
    es = view.element_size()
    aligned = view.data_ptr() % 16 == 0
    if layout == "contiguous":
        assert view.is_contiguous() and aligned
    elif layout == "padded":
        assert view.stride(0) == N + 8 and aligned
    elif layout == "misaligned":
        assert view.stride(0) % 2 == 1 and view.data_ptr() % 16 == es
    else:
        assert view.stride(0) % 8 == 0 and view.data_ptr() % 16 == es
    return view


def n_frames(L, w, s):
    return O.frame_count(L, w, s)


def ragged_lengths(N, w, s):
    """N; L < w (no frame); L == w (one frame); an odd and an even frame count that end mid-hop; N - 1."""
    T = n_frames(N, w, s)
    t_odd = max(3, (T // 2) | 1)
    L_odd = w + (t_odd - 1) * s + s // 2
    L_even = w + t_odd * s + s - 1
    lens = [N, w - 1, w, L_odd, L_even, N - 1]
    assert n_frames(w - 1, w, s) == 0 and n_frames(w, w, s) == 1
    assert n_frames(L_odd, w, s) % 2 == 1 and n_frames(L_even, w, s) % 2 == 0 and L_even < N - 1
    return lens


# ---------------------------------------------------------------------------------------------- feature matrix
# (fs, w, s, N), chosen per code-path flag:
#   pair: step == w/2 on a window of whole 160-sample halves (shared halves) and not; 512 / 1024 never share
#   CTA on 80-multiple windows: step % 8 == 0 (8-sample runs), even but not a multiple of 8, odd
#   solo: 882 / 441, 400 / 160, 600 / 150
FEATURE_CONFIGS = [
    (16000, 800, 400, 24000),      # pair shared, CTA runs
    (16000, 800, 320, 24000),      # pair not shared, CTA runs
    (16000, 800, 202, 16000),      # CTA even hop
    (16000, 640, 320, 24000),      # pair shared, CTA runs
    (16000, 640, 162, 16000),      # pair not shared, CTA even hop
    (16000, 480, 240, 24000),      # pair shared, CTA runs
    (16000, 320, 161, 16000),      # CTA odd hop, pair not shared
    (16000, 512, 256, 24000),      # pair (no sharing at 512)
    (48000, 960, 480, 48000),      # pair shared
    (16000, 1024, 300, 24000),     # pair not shared
    (44100, 882, 441, 44096),      # solo, CTA odd hop on a non-80-multiple window
    (16000, 400, 160, 24000),      # solo, CTA runs
    (8000, 600, 150, 16000),       # solo, CTA even hop (600 is not an 80-multiple: no runs)
    (16000, 400, 133, 16000),      # solo, CTA odd hop
]
N_CLIPS = 6


def check_base_and_deltas(got, ref, K, what):
    """The 34 base rows against the oracle at the standard tolerance; delta rows (if any) must be the first difference
    of the kernel's own base rows (0 in column 0).  One float32-vs-float64 tie of spectral_rolloff moves the base row
    and two delta columns, three quantum flips that the two-flip budget of a clip of under ~750 frames does not
    allow (measured: pair kernel 800 / 320 float32, generic kernel 320 / 161 int16); counted on the base rows it is
    one flip."""
    check_features(got[:34], ref[:34], K, what)
    if got.shape[0] == 68:
        base = got[:34].astype(np.float64)
        assert not got[34:, 0].any(), what + ": delta column 0 is not zero"
        diff = base[:, 1:] - base[:, :-1]
        bad = np.abs(got[34:, 1:] - diff) > 1e-6 * (np.abs(base[:, 1:]) + np.abs(base[:, :-1]))
        assert not bad.any(), "%s: delta rows are not the first difference of the base rows at %s" % (what, np.argwhere(bad)[:5].tolist())


@pytest.mark.parametrize("fs,w,s,N", FEATURE_CONFIGS, ids=["%d-%d-%d" % c[:3] for c in FEATURE_CONFIGS])
def test_feature_matrix(P, plans, fs, w, s, N):
    clips16 = np.stack([O.synth_clip(500 + 17 * i + w, N, fs) for i in range(N_CLIPS)])
    lens = ragged_lengths(N, w, s)
    T = n_frames(N, w, s)
    t_stride = T + 5
    K = w // 2
    refs = {}

    def ref(dtype, i, L):
        if (dtype, i, L) not in refs:
            x = as_dtype(clips16[i], dtype)[:L]
            refs[dtype, i, L] = O.feature_extraction(x, fs, w, s)[0] if L >= w else None
        return refs[dtype, i, L]

    import torch
    for dtype in ("int16", "float32"):
        clips = as_dtype(clips16, dtype)
        for ragged in (False, True):
            lengths = lens if ragged else None
            d_len = torch.tensor(lens, dtype=torch.int64, device="cuda") if ragged else None
            Ls = lens if ragged else [N] * N_CLIPS
            for layout in LAYOUTS:
                d = device_clips(clips, lengths, layout, seed=w + s)
                for deltas in (True, False):
                    F = 68 if deltas else 34
                    for kind in feature_kernels(w):
                        what = "%s kernel, %s %s, %s, deltas=%s, fs=%d w=%d s=%d" % (
                            KIND_NAME[kind], dtype, layout, "ragged" if ragged else "full", deltas, fs, w, s)
                        out = nan_filled((N_CLIPS, F, t_stride))
                        P.feature_extraction_batch(d, fs, w, s, deltas=deltas, out=out, lengths=d_len, plan=plans(fs, w, s, kind))
                        got = out.cpu().numpy()
                        bits = got.view(np.uint32)
                        for i, L in enumerate(Ls):
                            Ti = n_frames(L, w, s)
                            assert (bits[i, :, Ti:] == NAN_BITS).all(), \
                                "%s: clip %d (L=%d) has writes in columns [%d, %d)" % (what, i, L, Ti, t_stride)
                            if Ti == 0:
                                continue
                            assert not np.isnan(got[i, :, :Ti]).any(), "%s: clip %d (L=%d) has unwritten columns" % (what, i, L)
                            check_base_and_deltas(got[i, :, :Ti], ref(dtype, i, L), K, "%s, clip %d, L=%d" % (what, i, L))


# ---------------------------------------------------------------------------------------------- row modes
ROW_CONFIGS = [(16000, 800, 400), (16000, 800, 200), (44100, 882, 441), (16000, 400, 160), (8000, 600, 300),
               (16000, 320, 160), (16000, 480, 240), (16000, 640, 320), (16000, 640, 161), (16000, 512, 256),
               (48000, 960, 480), (16000, 1024, 512)]


# Spectrogram entries are |X|/K of frames normalised to peak 1 (typically 1e-3 .. 4e-2).  The generic kernel's float32
# transform of float32 clips was measured 1.3e-7 .. 1.6e-7 off on single entries (320 / 160, 640 / 161, 512 / 256;
# 4e-6 of the largest entry), just above the 1e-7 the int16 golden tests use, and still 50x below parity.ATOL.
SPEC_ATOL = 2e-7


def chroma_tail(N, w, s):
    """Samples the last chromagram frame gets (ShortTermFeatures.py:349: frames start at w, w + s, ... < N - s)."""
    p_last = w + s * ((N - s - 1 - w) // s)
    return N - p_last


def row_lengths(fs, w, s):
    """About one second with the last chromagram frame clipped (but >= K samples, which the reference accepts), and
    one with it whole -- when the hop allows it (the last frame is always clipped when s < w / 2).  Multiples of 8
    samples come first, so that padded clips keep the CTA kernel's 8-sample runs."""
    out = []
    cands = sorted(range(fs, fs + 4 * w), key=lambda n: (n % 8 != 0, n))
    for clipped in (True, False):
        for N in cands:
            r = chroma_tail(N, w, s)
            if (w // 2 <= r < w) if clipped else (r >= w):
                out.append(N)
                break
    return out


@pytest.mark.parametrize("fs,w,s", ROW_CONFIGS, ids=["%d-%d-%d" % c for c in ROW_CONFIGS])
def test_row_matrix(P, plans, fs, w, s):
    Ns = row_lengths(fs, w, s)
    assert Ns and (s < w // 2 or len(Ns) == 2)
    for N in Ns:
        clips16 = np.stack([O.synth_clip(700 + 11 * i + w, N, fs) for i in range(3)])
        for dtype in ("int16", "float32"):
            clips = as_dtype(clips16, dtype)
            sp_ref = [O.spectrogram(c, fs, w, s)[0] for c in clips]
            ch_ref = [O.chromagram(c, fs, w, s)[0] for c in clips]
            for layout in LAYOUTS:
                d = device_clips(clips, None, layout, seed=N)
                for kind in row_kernels(w):
                    pl = plans(fs, w, s, kind)
                    what = "%s kernel, %s %s, fs=%d w=%d s=%d N=%d (last chroma frame %d samples)" % (
                        KIND_NAME[kind], dtype, layout, fs, w, s, N, chroma_tail(N, w, s))
                    sp = P.spectrogram_batch(d, fs, w, s, plan=pl).cpu().numpy()
                    ch = P.chromagram_batch(d, fs, w, s, plan=pl).cpu().numpy()
                    for i in range(3):
                        check_close(sp[i], sp_ref[i], "spectrogram, " + what, atol=SPEC_ATOL)
                        check_close(ch[i], ch_ref[i], "chromagram, " + what, atol=1e-6)


def test_row_lengths_cover_both_chroma_ends():
    clipped = whole = 0
    for fs, w, s in ROW_CONFIGS:
        for N in row_lengths(fs, w, s):
            r = chroma_tail(N, w, s)
            clipped += r < w
            whole += r >= w
    assert clipped >= len(ROW_CONFIGS) and whole >= 8


def test_spectrogram_out_fully_written(P, plans):
    """spectrogram_batch(out=...) writes every element: the rows the reference allocates but never fills are 0."""
    for fs, w, s in ROW_CONFIGS:
        N = fs + 3 * s // 2
        clips = np.stack([O.synth_clip(900 + i, N, fs) for i in range(3)])
        import torch
        d = torch.from_numpy(clips).cuda()
        refs = [O.spectrogram(c, fs, w, s)[0] for c in clips]
        R, valid = refs[0].shape[0], len(range(w, N - w + 1, s))
        assert 0 < valid < R
        for kind in row_kernels(w):
            out = nan_filled((3, R, w // 2))
            P.spectrogram_batch(d, fs, w, s, plan=plans(fs, w, s, kind), out=out)
            got = out.cpu().numpy()
            what = "%s kernel, fs=%d w=%d s=%d" % (KIND_NAME[kind], fs, w, s)
            assert not np.isnan(got).any(), what + ": elements left unwritten"
            assert (got[:, valid:] == 0).all(), what + ": rows past the last frame are not zero"
            for i in range(3):
                check_close(got[i], refs[i], "spectrogram into out, " + what, atol=1e-7)


# ---------------------------------------------------------------------------------------------- adversarial clips
ADV_CONFIGS = [(16000, 800, 400), (44100, 882, 441), (8000, 400, 200), (16000, 512, 256)]
ADV_N = 16000


def integer_mean_ties(fs, N):
    """Mean exactly 7 with runs of samples at 7 between noise of both signs (ties count half a crossing)."""
    x = O.synth_clip(31, N, fs).astype(np.int64) // 2
    tie = np.zeros(N, bool)
    for k in range(0, N - 6, 23):
        tie[k:k + 1 + k % 5] = True
    x[tie] = 0
    free = np.nonzero(~tie)[0]
    r = int(x.sum())
    x[free] -= r // len(free)                          # the remainder (0 <= rem < len(free)) one unit at a time
    x[free[:r - (r // len(free)) * len(free)]] -= 1
    x += 7
    assert x.sum() == 7 * N and x.min() >= -32768 and x.max() <= 32767
    ties = x == 7
    assert ties.sum() > N // 20
    idx = np.nonzero(ties[1:-1])[0] + 1
    same = np.sign(x[idx - 1] - 7) * np.sign(x[idx + 1] - 7)
    assert (same > 0).any() and (same < 0).any()       # ties between same-sign and opposite-sign neighbours
    return x.astype(np.int16)


def integer_mean_ties_f32(fs, N):
    """Float variant: x * 0.5 + 3.25 is exact in float32, and so is its mean, 6.75."""
    x = integer_mean_ties(fs, N).astype(np.float32) * np.float32(0.5) + np.float32(3.25)
    assert x.astype(np.float64).sum() / N == 6.75 and (x == np.float32(6.75)).sum() > N // 20
    return x


def full_scale(fs, N):
    """A hard-clipped sine plus noise that reaches both -32768 and 32767."""
    t = np.arange(N) / fs
    rng = np.random.default_rng(5)
    x = np.clip(np.round(45000 * np.sin(2 * np.pi * 220.0 * t) + 2000 * rng.standard_normal(N)), -32768, 32767).astype(np.int16)
    assert x.min() == -32768 and x.max() == 32767
    return x


def negative_excursion(fs, N):
    """Sparse large negative spikes: mean - min > max - mean, so the negative side sets the scale."""
    x = O.synth_clip(33, N, fs).astype(np.int64) // 4
    x[::997] = -30000
    m = x.mean()
    assert m - x.min() > 3 * (x.max() - m)
    return x.astype(np.int16)


def large_dc(fs, N):
    """Mean about 20000 with +-3000 of signal on top."""
    t = np.arange(N) / fs
    rng = np.random.default_rng(6)
    ac = np.clip(2000 * np.sin(2 * np.pi * 330.0 * t) + 300 * rng.standard_normal(N), -3000, 3000)
    x = np.round(20000 + ac).astype(np.int16)
    assert abs(x.mean() - 20000) < 50 and np.abs(x.astype(np.int64) - 20000).max() <= 3000
    return x


def large_dc_f32(fs, N):
    x = (O.synth_clip(34, N, fs).astype(np.float64) / 32768.0 + 1e3).astype(np.float32)
    assert abs(x.mean() - 1e3) < 0.01
    return x


SWEEP_PEAKS = (1e-6, 1e-3, 1.0, 3e4)


def scaled(peak):
    def build(fs, N):
        x = O.synth_clip(35, N, fs).astype(np.float64)
        x = (x * (peak / np.abs(x).max())).astype(np.float32)
        assert abs(np.abs(x.astype(np.float64)).max() / peak - 1) < 1e-6
        return x
    return build


ADV_CLIPS = [("integer mean with ties", integer_mean_ties), ("float32 exact mean with ties", integer_mean_ties_f32),
             ("full scale", full_scale), ("full scale float32", lambda fs, N: full_scale(fs, N).astype(np.float32) * 0.37),
             ("negative excursion", negative_excursion),
             ("negative excursion float32", lambda fs, N: negative_excursion(fs, N).astype(np.float32) * 1.9 - 40),
             ("large DC", large_dc), ("large DC float32", large_dc_f32)] + \
            [("float32 peak %g" % p, scaled(p)) for p in SWEEP_PEAKS]


@pytest.mark.parametrize("name,build", ADV_CLIPS, ids=[c[0].replace(" ", "_") for c in ADV_CLIPS])
def test_adversarial_clips(P, plans, name, build):
    import torch
    for fs, w, s in ADV_CONFIGS:
        x = build(fs, ADV_N)
        ref = O.feature_extraction(x, fs, w, s)[0]
        d = torch.from_numpy(np.ascontiguousarray(x)[None]).cuda()
        for kind in feature_kernels(w):
            got = P.feature_extraction_batch(d, fs, w, s, plan=plans(fs, w, s, kind))[0].cpu().numpy()
            check_features(got, ref, w // 2, "%s: %s kernel, fs=%d w=%d s=%d" % (name, KIND_NAME[kind], fs, w, s))


def test_quiet_float_clips_are_not_scale_invariant():
    """The reference's +1e-10 (after /2**15) sets the scale of clips whose peak is near 2**15 * 1e-10: the same waveform
    at peak 1e-6 and at peak 1 gives different features (test_adversarial_clips holds the GPU to both)."""
    fs, w, s = 16000, 800, 400
    quiet = O.feature_extraction(scaled(1e-6)(fs, ADV_N), fs, w, s)[0]
    loud = O.feature_extraction(scaled(1.0)(fs, ADV_N), fs, w, s)[0]
    louder = O.feature_extraction(scaled(3e4)(fs, ADV_N), fs, w, s)[0]
    check_features(louder, loud, w // 2, "peak 3e4 vs peak 1")          # 1e-10 is a 3e-6 relative change at peak 1
    assert np.abs(quiet[1] / loud[1] - 1).min() > 0.5                     # energy
    assert np.abs(quiet[8] - loud[8]).min() > 0.1                         # mfcc_1


# ---------------------------------------------------------------------------------------------- large batch
def test_large_batch(P, plans):
    """40000 clips: clip statistics run in chunks of 32768 clips; clips on both sides of the boundary, each distinct
    (a shifted waveform plus its own DC) with its own length, against the oracle."""
    import torch
    B, N = 40000, 2000
    i = np.arange(B)
    base = O.synth_clip(41, 8192, 16000).astype(np.int32) // 2
    idx = (np.arange(N)[None, :] + (37 * i)[:, None]) % base.shape[0]
    dc = (i * 7919) % 2001 - 1000
    clips = (base[idx] + dc[:, None]).astype(np.int16)
    lens = 900 + (i * 104729) % 1101                  # at least one frame of either window
    check = sorted({0, 1, 32767, 32768, 32769, B - 1} | set(np.random.default_rng(3).integers(0, B, 5).tolist()))
    assert len(set(lens[[0, 1, 32767, 32768, 32769]].tolist())) == 5 and len(set(dc[[0, 1, 32767, 32768, 32769]].tolist())) == 5
    d16 = torch.from_numpy(clips).cuda()
    d_len = torch.from_numpy(lens.astype(np.int64)).cuda()
    for dtype in ("int16", "float32"):
        d = d16 if dtype == "int16" else d16.to(torch.float32) * 0.613 + 2.5
        host = {c: d[c].cpu().numpy() for c in check}
        for fs, w, s in ((16000, 800, 400), (44100, 882, 441)):
            refs = {c: O.feature_extraction(host[c][:lens[c]], fs, w, s)[0] for c in check}
            for kind in feature_kernels(w):
                out = P.feature_extraction_batch(d, fs, w, s, lengths=d_len, plan=plans(fs, w, s, kind))
                assert out.shape == (B, 68, n_frames(N, w, s))
                for c in check:
                    Tc = refs[c].shape[1]
                    got = out[c].cpu().numpy()
                    check_features(got[:, :Tc], refs[c], w // 2, "%s kernel, %s, fs=%d w=%d s=%d, clip %d of %d (L=%d)" % (
                        KIND_NAME[kind], dtype, fs, w, s, c, B, lens[c]))
                    assert not got[:, Tc:].any()
                del out
