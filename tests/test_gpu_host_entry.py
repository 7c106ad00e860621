"""GPU: the host-buffer entry points (b200aa_*_host: what the drop-in ShortTermFeatures / MidTermFeatures calls and
HostPipeline run) and concurrent callers.

- The chunked three-stream form of b200aa_st_features_host, on both sides of its switch-over and of every chunk
  boundary, for int16 and float32 clips, with and without deltas, bit for bit against the device-resident path.
- One plan's grow-only workspaces through a sequence of calls that grows, shrinks and reuses every one of them.
- Threads on their own streams sharing cached plans (pair, solo, big-window generic), a plan pinned to the CTA kernel,
  the drop-in host calls and the chunked pipeline: every result equals the same call made alone.
"""
import threading

import numpy as np
import pytest

from oracle import st_oracle as O
from tests.parity import check_features

pytestmark = pytest.mark.gpu

FS, W, S = 16000, 800, 400
PIPE_N = 1 << 21                                   # T = 5241; a chunk is 8 int16 or 4 float32 clips (32 MiB)
NAN_BITS = np.uint32(0x7FC0DEAD)


@pytest.fixture(scope="module")
def P():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import pyaudioanalysis_b200 as pkg
    pkg.ShortTermFeatures.PRINT_SPECTROGRAM_SHAPE = False
    pkg.MidTermFeatures.VERBOSE = False
    return pkg


def distinct_clips(seed, n_clips, n, dtype):
    """n_clips different clips of n samples: windows of one long clip at distinct shifts, each with its own DC offset
    (float32: also its own scale)."""
    base = O.synth_clip(seed, n + 4099 * n_clips, FS).astype(np.int32)
    out = np.empty((n_clips, n), dtype=dtype)
    for i in range(n_clips):
        x = base[4099 * i:4099 * i + n] + (37 * i - 500)
        if dtype == np.int16:
            out[i] = np.clip(x, -32768, 32767)
        else:
            out[i] = x.astype(np.float32) * np.float32(1.0 / (3000.0 + 250.0 * i))
    return out


def nan_filled(shape):
    return np.full(shape, NAN_BITS, dtype=np.uint32).view(np.float32)


def launches():
    from pyaudioanalysis_b200 import _lib
    return _lib.lib().b200aa_launch_count()


def device_features(P, clips, deltas, fs=FS, w=W, s=S, plan=None):
    import torch
    return P.feature_extraction_batch(torch.from_numpy(np.ascontiguousarray(clips)).cuda(), fs, w, s, deltas=deltas,
                                      plan=plan).cpu().numpy()


@pytest.mark.parametrize("dtype,sizes", [(np.int16, (15, 16, 17, 29)), (np.float32, (7, 8, 9, 14))], ids=["int16", "float32"])
def test_chunked_pipeline(P, dtype, sizes):
    """Batches just below two chunks (one stream), at two, just above, and over three streams with one reused; deltas
    on and off.  The output buffer has more rows than the batch and a NaN payload: rows past the batch keep it bit for
    bit.  Launch counts show which form ran."""
    from pyaudioanalysis_b200.hostpipe import HostPipeline
    chunk = (32 << 20) // (PIPE_N * np.dtype(dtype).itemsize)
    n_max = max(sizes)
    clips = distinct_clips(710 if dtype == np.int16 else 711, n_max, PIPE_N, dtype)
    oracle = {}

    def ref(i):
        if i not in oracle:
            oracle[i] = O.feature_extraction(clips[i], FS, W, S)[0]
        return oracle[i]

    for deltas in (False, True):
        pipe = HostPipeline(FS, W, S, PIPE_N, max_clips=n_max, deltas=deltas, dtype=dtype)
        assert pipe.T == 5241
        pipe.h_in[:] = clips
        before = launches()
        pipe.run(pipe.h_in[:1])
        per_call = launches() - before
        for B in sizes:
            out = nan_filled((B + 3, pipe.F, pipe.T))
            before = launches()
            got = pipe.run(pipe.h_in[:B], out=out)
            n_launch = launches() - before
            chunks = -(-B // chunk)
            assert n_launch == (per_call * chunks if B >= 2 * chunk else per_call), (B, n_launch, per_call)
            assert got.shape == (B, pipe.F, pipe.T)
            assert not np.isnan(out[:B]).any(), "B %d: rows of the batch not fully written" % B
            assert (out[B:].view(np.uint32) == NAN_BITS).all(), "B %d: rows past the batch were written" % B
            dev = device_features(P, clips[:B], deltas)
            assert np.array_equal(out[:B], dev), "B %d deltas %d: host pipeline differs from the device path" % (B, deltas)
            edges = {0, B - 1} | {k for a in range(chunk, B, chunk) for k in (a - 1, a)}
            for i in sorted(edges):
                check_features(out[i], ref(i)[:pipe.F], W // 2, "B %d clip %d deltas %d" % (B, i, deltas))


def test_workspace_reuse(P):
    """One cached plan's workspaces grown, shrunk and reused by a sequence of different host calls; each result equals
    the device path bit for bit."""
    import torch
    from pyaudioanalysis_b200.batch import chromagram_batch, mid_feature_extraction_batch, spectrogram_batch
    from pyaudioanalysis_b200.hostpipe import HostPipeline
    ST, MT = P.ShortTermFeatures, P.MidTermFeatures

    def dev(x):
        return torch.from_numpy(np.ascontiguousarray(x)).cuda().reshape(1, -1)

    x10 = O.synth_clip(720, 10 * FS, FS)
    assert np.array_equal(ST.feature_extraction(x10, FS, W, S)[0], device_features(P, x10[None], True)[0])
    x60 = O.synth_clip(721, 60 * FS, FS)
    assert np.array_equal(ST.spectrogram(x60, FS, W, S)[0], spectrogram_batch(dev(x60), FS, W, S)[0].cpu().numpy())
    x3 = O.synth_clip(722, 3 * FS, FS)
    assert np.array_equal(ST.chromagram(x3, FS, W, S)[0], chromagram_batch(dev(x3), FS, W, S)[0].cpu().numpy())
    x30 = O.synth_clip(723, 30 * FS, FS).astype(np.float32) * np.float32(1e-4) + np.float32(0.25)
    mid, st, _ = MT.mid_feature_extraction(x30, FS, FS, FS // 2, W, S)
    mid_d, st_d = mid_feature_extraction_batch(dev(x30), FS, FS, FS // 2, W, S)
    assert np.array_equal(mid, mid_d[0].cpu().numpy()) and np.array_equal(st, st_d[0].cpu().numpy())
    x1 = O.synth_clip(724, FS, FS)
    assert np.array_equal(ST.feature_extraction(x1, FS, W, S)[0], device_features(P, x1[None], True)[0])
    clips = distinct_clips(725, 17, PIPE_N, np.int16)
    for deltas in (False, True):
        pipe = HostPipeline(FS, W, S, PIPE_N, max_clips=17, deltas=deltas)
        assert np.array_equal(pipe.run(clips), device_features(P, clips, deltas))
    two = distinct_clips(726, 2, PIPE_N, np.float32)
    pipe = HostPipeline(FS, W, S, PIPE_N, max_clips=2, dtype=np.float32)
    assert np.array_equal(pipe.run(two), device_features(P, two, True))


def test_concurrent_callers(P):
    """Serial results first; then at once: 6 threads on their own streams (30 iterations each, distinct batches) sharing
    the cached 800 / 400 (pair kernel), 882 / 441 (solo kernel) and 44100 / 44100 (big-window generic kernel, stream-
    ordered scratch) plans and one 800 / 400 plan pinned to the CTA kernel, over 64 launches per plan so the ring of
    work-counter slots wraps; 2 threads calling the drop-in feature_extraction / mid_feature_extraction; 1 thread running
    the chunked host pipeline.  Every output equals its serial result bit for bit."""
    import torch
    from pyaudioanalysis_b200._lib import Plan, get_plan
    from pyaudioanalysis_b200.hostpipe import HostPipeline
    n_threads, iters = 6, 30
    cta = Plan(FS, W, S).prefer_kernel(1)
    assert cta.kernel_kind() == 1
    assert get_plan(FS, W, S).kernel_kind() == 2 and get_plan(44100, 882, 441).kernel_kind() == 3
    b16 = O.synth_clip(730, 2 * FS + 97 * n_threads * iters + 64, FS)
    b44 = O.synth_clip(731, 2 * 44100 + 97 * n_threads * iters + 64, 44100)

    def batch(base, j, n):
        return torch.from_numpy(np.stack([base[97 * j + 31 * k:97 * j + 31 * k + n] for k in range(2)])).cuda()

    # per iteration: the pair plan, then the solo or the CTA plan, and every third iteration the big-window plan
    work = []
    for t in range(n_threads):
        for i in range(iters):
            j = t * iters + i
            calls = [(batch(b16, j, 2 * FS), FS, W, S, None),
                     (batch(b44, j, 44100), 44100, 882, 441, None) if i % 2 else (batch(b16, j, 2 * FS), FS, W, S, cta)]
            if i % 3 == 0:
                calls.append((batch(b44, j, 2 * 44100), 44100, 44100, 44100, None))
            work.append(calls)
    serial = [[P.feature_extraction_batch(x, fs, w, s, plan=pl).cpu().numpy() for x, fs, w, s, pl in calls] for calls in work]
    drop_st = [O.synth_clip(740 + j, FS + 13 * j, FS) for j in range(iters)]
    drop_mid = [O.synth_clip(780 + j, 3 * FS + 29 * j, FS) for j in range(iters)]
    serial_st = [P.ShortTermFeatures.feature_extraction(x, FS, W, S)[0] for x in drop_st]
    serial_mid = [P.MidTermFeatures.mid_feature_extraction(x, FS, FS, FS // 2, W, S)[0] for x in drop_mid]
    pipe_n, pipe_b = 1 << 20, 33                   # chunks of 16 clips: three streams
    pipe = HostPipeline(FS, W, S, pipe_n, max_clips=pipe_b)
    pipe_in = [distinct_clips(750 + r, pipe_b, pipe_n, np.int16) for r in range(2)]
    serial_pipe = [pipe.run(x, out=np.empty((pipe_b, 68, pipe.T), np.float32)).copy() for x in pipe_in]
    torch.cuda.synchronize()

    errors = []

    def guarded(fn):
        def run():
            try:
                fn()
            except BaseException as e:          # re-raised in the main thread
                errors.append(e)
        return run

    def stream_worker(t):
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            for i in range(iters):
                j = t * iters + i
                for k, (x, fs, w, st, pl) in enumerate(work[j]):
                    got = P.feature_extraction_batch(x, fs, w, st, plan=pl).cpu().numpy()
                    assert np.array_equal(got, serial[j][k]), "thread %d iteration %d call %d (%d / %d)" % (t, i, k, w, st)

    def drop_st_worker():
        for j, x in enumerate(drop_st):
            assert np.array_equal(P.ShortTermFeatures.feature_extraction(x, FS, W, S)[0], serial_st[j]), "drop-in st %d" % j

    def drop_mid_worker():
        for j, x in enumerate(drop_mid):
            got = P.MidTermFeatures.mid_feature_extraction(x, FS, FS, FS // 2, W, S)[0]
            assert np.array_equal(got, serial_mid[j]), "drop-in mid %d" % j

    def pipe_worker():
        for r, x in enumerate(pipe_in):
            got = pipe.run(x, out=np.empty((pipe_b, 68, pipe.T), np.float32))
            assert np.array_equal(got, serial_pipe[r]), "host pipeline run %d" % r

    fns = [lambda t=t: stream_worker(t) for t in range(n_threads)] + [drop_st_worker, drop_mid_worker, pipe_worker]
    threads = [threading.Thread(target=guarded(fn), daemon=True) for fn in fns]
    for th in threads:
        th.start()
    for th in threads:
        th.join(timeout=600)
    assert not any(th.is_alive() for th in threads), "a thread did not finish within 600 s"
    if errors:
        raise errors[0]
