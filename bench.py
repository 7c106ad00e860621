#!/usr/bin/env python
"""bench.py -- short-term feature_extraction throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[1] -- 1000 synthetic 16 kHz mono int16 10 s clips per
GPU, window/step 50/25 ms, full 68-row short-term feature matrix.  One "step" = the whole hot path
over the batch: clip statistics (kernel 0) + fused short-term features (kernel 1); for N > 1 every
rank's [clips, 68, T] block is pushed by the copy engines into rank 0's peer-mapped gather buffer
(NVLink, b200aa_peer_buffer_* / b200aa_peer_copy) under the next step's kernels, all pushes inside the timed
region (`scaling_detail` also gives the step without any gather, with a plain NCCL gather, and with the
gather fused into the kernel's stores).
Prints ONE JSON line (rank 0).  `value` = frames/s with inputs resident in HBM; `e2e` = the same metric
through the C ABI's host entry point b200aa_st_features_host (pinned host clips in, pinned host features
out, copies inside the timed region); `roofline` = algorithmic bytes / kernel time of the fused kernel
against the measured HBM peak (plus the FP32-issue fraction of the committed ncu capture);
`cpu_baseline` = the unmodified reference (staged under oracle/_ref by oracle/make_ref.py) on the host
cores, one single-threaded process per physical core, bounded sample.
`--dump-outputs DIR` writes the feature matrices of the last timed step (rank 0: the gathered ones) for a fixed, seeded
sample of DUMP_CLIPS clips as DIR/features.npy (float32 [DUMP_CLIPS, 68, T], 55.6 MB); the clips are generated from fixed
seeds, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import multiprocessing as mp
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FS, WINDOW, STEP, CLIP_SAMPLES, CLIPS_PER_GPU = 16000, 800, 400, 160000, 1000
FRAMES_PER_CLIP = (CLIP_SAMPLES - WINDOW) // STEP + 1            # 399
DUMP_CLIPS = 512                                                  # --dump-outputs: 512 x 68 x 399 float32 = 55.6 MB
ALG_BYTES_PER_CLIP = 2 * CLIP_SAMPLES + 4 * 68 * FRAMES_PER_CLIP   # 428 528 (SURVEY.md 8d)
METRIC = "audio frames/sec short-term feature_extraction @16kHz 50/25ms"
WORKLOAD = "1000 synthetic 16 kHz mono int16 10 s clips per GPU, win/step 50/25 ms, 68 short-term features (BASELINE configs[1])"
# identical in both arms (the driver compares the dicts); arm-specific detail goes to `detail`
CONFIG = {"workload": WORKLOAD, "fs": FS, "window": WINDOW, "step": STEP, "clip_samples": CLIP_SAMPLES,
          "clips_per_gpu": CLIPS_PER_GPU, "frames_per_clip": FRAMES_PER_CLIP, "n_features": 68,
          "parallelism": "clips sharded per GPU, feature matrices gathered on rank 0"}


# ----------------------------------------------------------------------------- CPU baseline (unmodified reference)
_PIN_ENV = {"OMP_NUM_THREADS": "1", "MKL_NUM_THREADS": "1", "OPENBLAS_NUM_THREADS": "1", "NUMEXPR_NUM_THREADS": "1",
            "VECLIB_MAXIMUM_THREADS": "1"}
_cpu_state = {}


def physical_cores():
    """One logical CPU per physical core among the CPUs this process may run on."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
    except AttributeError:
        return list(range(os.cpu_count() or 1))
    seen, out = set(), []
    for c in allowed:
        try:
            with open("/sys/devices/system/cpu/cpu%d/topology/thread_siblings_list" % c) as f:
                key = f.read().strip()
        except OSError:
            key = str(c)
        if key not in seen:
            seen.add(key)
            out.append(c)
    return out


def cpu_quota():
    """CPUs' worth of time the container may use per period (cgroup v2 cpu.max / v1 cfs quota), or None if unlimited."""
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, p = f.read().split()
            return None if q == "max" else float(q) / float(p)
    except (OSError, ValueError):
        pass
    try:
        with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
            q = float(f.read())
        with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
            p = float(f.read())
        return None if q <= 0 else q / p
    except (OSError, ValueError):
        return None


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def _cpu_init(core_q, kind):
    """Worker start: one process per physical core, BLAS pools off, the implementation imported once."""
    os.environ.update(_PIN_ENV)
    try:
        os.sched_setaffinity(0, {core_q.get_nowait()})
    except Exception:
        pass
    try:
        from threadpoolctl import threadpool_limits
        _cpu_state["tp"] = threadpool_limits(1)
    except Exception:
        pass
    from oracle import st_oracle as O
    _cpu_state["clips"] = [O.synth_clip(1000 * (os.getpid() % 977) + i, CLIP_SAMPLES, FS) for i in range(4)]   # outside the timed work
    if kind == "reference":
        import warnings
        warnings.simplefilter("ignore")
        from oracle.ref_import import load_reference
        S = load_reference(staged_ok=True)[0]
        _cpu_state["fe"] = lambda x: S.feature_extraction(x, FS, WINDOW, STEP)[0]
    else:
        _cpu_state["fe"] = lambda x: O.feature_extraction_loop(x, FS, WINDOW, STEP, deltas=True, tables_per_frame=True)[0]


def _cpu_worker(args):
    idx, n_clips = args
    frames = 0
    for i in range(n_clips):
        frames += _cpu_state["fe"](_cpu_state["clips"][(idx + i) % 4]).shape[1]
    return frames


def cpu_baseline(target_seconds=12.0, steps=1, warmup=0):
    """Time the reference's own feature_extraction on the host cores.

    `steps` timed passes (after `warmup` untimed ones) over a bounded sample of the workload: every pass runs `per`
    ten-second clips on each of `cores` single-threaded processes (one per physical core), `per` chosen from a
    one-clip probe so that the timed passes together take about `target_seconds`.
    Returns (cpu_baseline dict, frames, seconds) over the timed passes.
    """
    from oracle.ref_import import reference_available, staged_available
    kind = "reference" if (staged_available() or reference_available()) else "port"
    cores = physical_cores()
    quota = cpu_quota()
    if quota is not None and quota < len(cores):          # a throttled container: more processes than CPUs only add noise
        cores = cores[:max(1, int(quota))]
    if len(cores) > 128:
        cores = cores[:128]
    n = len(cores)
    os.environ.update(_PIN_ENV)            # inherited by the spawned workers before NumPy loads its BLAS
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    for c in cores:
        q.put(c)
    with ctx.Pool(n, initializer=_cpu_init, initargs=(q, kind)) as pool:
        pool.map(_cpu_worker, [(900 + c, 0) for c in range(n)], chunksize=1)      # start workers / import
        pool.apply(_cpu_worker, ((7, 1),))                                        # one clip on one process, the others idle:
        t0 = time.perf_counter()                                                  # the per-core rate without any contention
        single = pool.apply(_cpu_worker, ((8, 2),)) / (time.perf_counter() - t0)
        t0 = time.perf_counter()
        pool.map(_cpu_worker, [(c, 1) for c in range(n)], chunksize=1)            # probe: one clip per worker (also warm-up)
        probe = time.perf_counter() - t0
        per = max(1, int(target_seconds / max(steps, 1) / max(probe, 1e-3)))
        per = min(per, 32)
        for w in range(warmup):
            pool.map(_cpu_worker, [(5000 + 64 * w + c, 1) for c in range(n)], chunksize=1)
        frames, dt = 0, 0.0
        for k in range(max(steps, 1)):
            t0 = time.perf_counter()
            frames += sum(pool.map(_cpu_worker, [(100 + 64 * k + c, per) for c in range(n)], chunksize=1))
            dt += time.perf_counter() - t0
    what = ("the unmodified reference ShortTermFeatures.feature_extraction (oracle/_ref, staged by oracle/make_ref.py)"
            if kind == "reference" else "oracle.feature_extraction_loop (port with the reference's cost profile)")
    return {"value": frames / dt, "unit": "frames/s", "cores": n, "kind": kind, "cpu": cpu_model(),
            "threads_per_process": 1, "single_process_frames_per_s": single, "cgroup_cpu_quota": quota,
            "load_avg_1min": (os.getloadavg()[0] if hasattr(os, "getloadavg") else None),
            "sample": "%d pass(es) of %d clips of 10 s (%d frames in all), one single-threaded process pinned to each of %d "
                      "physical cores, %s, %.1f s wall" % (max(steps, 1), per * n, frames, n, what, dt)}, frames, dt


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    def __init__(self, index):
        self.index, self.samples, self.reasons, self.stop = index, [], set(), False
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80}
        while not self.stop:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.02)

    def __enter__(self):
        if self.nv:
            self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        if self.nv:
            self.t.join(timeout=1)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_facts():
    """Figures of the committed `ncu --set full` capture of the fused kernel (profiles/traffic.json): DRAM bytes per
    launch, warp instructions per launch, issue-slot utilisation.  Static by nature (a profiler cannot run inside
    the timed region); the file names the capture they come from."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


# ----------------------------------------------------------------------------- reference arm
def run_reference(args, rank, world):
    if rank != 0:
        return
    steps = args.steps
    cb, frames, dt = cpu_baseline(target_seconds=30.0, steps=steps, warmup=min(args.warmup, 3))
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "frames/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": CONFIG,
            "detail": "CPU arm: each step is a bounded sample of the workload (see cpu_baseline.sample); a rate on identical "
                      "clips and parameters",
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- our arm
def dump_clips(n_clips):
    """Indices of the clips --dump-outputs writes: a fixed, seeded sample (the same for every build)."""
    import numpy as np
    return np.sort(np.random.default_rng(0).choice(n_clips, DUMP_CLIPS, replace=False))


def synth_device_batch(torch, n_clips, seed, device):
    """Noise + three harmonics per clip, generated on the device (SURVEY.md 8d recipe, bulk variant)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = torch.empty((n_clips, CLIP_SAMPLES), dtype=torch.int16, device=device)
    t = torch.arange(CLIP_SAMPLES, device=device, dtype=torch.float32) / FS
    chunk = 100
    for c0 in range(0, n_clips, chunk):
        n = min(chunk, n_clips - c0)
        f0 = 80.0 + 920.0 * torch.rand((n, 1), generator=g, device=device)
        sig = 3000.0 * torch.randn((n, CLIP_SAMPLES), generator=g, device=device)
        for h in (1, 2, 3):
            sig += (6000.0 / h) * torch.sin(2 * torch.pi * h * f0 * t[None, :])
        out[c0:c0 + n] = sig.round().clamp(-32768, 32767).to(torch.int16)
    return out


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from pyaudioanalysis_b200 import numa
    try:
        full_affinity = os.sched_getaffinity(0)
    except AttributeError:
        full_affinity = None
    bound = numa.bind_to_gpu(local_rank)         # before any pinned allocation: staging buffers on the GPU's NUMA node
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import pyaudioanalysis_b200 as pkg
    from pyaudioanalysis_b200 import _lib
    from pyaudioanalysis_b200.hostpipe import HostPipeline
    from pyaudioanalysis_b200.dist import PeerGather
    L = _lib.lib()
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B = CLIPS_PER_GPU
    clips = synth_device_batch(torch, B, 1234 + rank, dev)
    plan = _lib.get_plan(FS, WINDOW, STEP, local_rank)
    T = FRAMES_PER_CLIP
    local_out = torch.empty((B, 68, T), dtype=torch.float32, device=dev)
    # N > 1: rank 0 owns a [world*B, 68, T] buffer that every rank maps over NVLink.  Default gather ("ce"): a rank's
    # kernels write a local block (double-buffered) and the copy engines push it into rank 0's buffer on a second
    # stream, under the kernels of the next step; all pushes complete inside the timed region.  "p2p_store": the kernel
    # stores straight into the mapped buffer; "nccl": torch.distributed.gather; "none": no gather.
    gathers = [PeerGather(world * B, 68, T, dst=0) for _ in range(2)] if world > 1 else None
    nccl_dst = [torch.empty((world, B, 68, T), dtype=torch.float32, device=dev)] if (world > 1 and rank == 0) else None
    local2 = [local_out, torch.empty_like(local_out)] if world > 1 else [local_out]
    copy_stream = torch.cuda.Stream(dev) if world > 1 else None

    ev = lambda: torch.cuda.Event(enable_timing=True)     # noqa: E731

    def timed(mode, steps, record_kernel=False):
        """`steps` passes in gather mode `mode` ('ce' | 'p2p_store' | 'none' | 'nccl'); returns (ms total max over ranks, kernel ms)."""
        ks, ke = [ev() for _ in range(steps)], [ev() for _ in range(steps)]
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        cur = torch.cuda.current_stream()
        pushed = [None, None]
        e0, e1 = ev(), ev()
        e0.record()
        for i in range(steps):
            norm = pkg.clip_stats(clips)
            if mode == "p2p_store" and world > 1:
                out = gathers[i % 2].view(rank * B, (rank + 1) * B)
            elif mode == "ce" and world > 1:
                if rank == 0:
                    out = gathers[i % 2].view(0, B)                 # the root's own block needs no copy
                else:
                    out = local2[i % 2]
                    if pushed[i % 2] is not None:
                        cur.wait_event(pushed[i % 2])               # the block's previous push must have left the buffer
            else:
                out = local_out
            ks[i].record()
            pkg.feature_extraction_batch(clips, FS, WINDOW, STEP, deltas=True, out=out, norm=norm, plan=plan)
            ke[i].record()
            if mode == "ce" and world > 1 and rank != 0:
                copy_stream.wait_event(ke[i])
                gathers[i % 2].push(out, rank * B, stream=copy_stream)
                pushed[i % 2] = torch.cuda.Event()
                pushed[i % 2].record(copy_stream)
            if mode == "nccl" and world > 1:
                dist.gather(local_out, [nccl_dst[0][r] for r in range(world)] if rank == 0 else None, dst=0)
        for p_ in pushed:
            if p_ is not None:
                cur.wait_event(p_)                                  # every push completes inside the timed region
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()          # all ranks' transfers have landed before the clock is read
        ms = e0.elapsed_time(e1)
        kms = sum(a.elapsed_time(b) for a, b in zip(ks, ke)) / steps
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), kms

    main_mode = "ce" if world > 1 else "none"
    timed(main_mode, max(3, args.warmup))
    launches0 = L.b200aa_launch_count()
    with ClockSampler(local_rank) as clk:
        ms_total, kernel_ms = timed(main_mode, args.steps)
        launches = L.b200aa_launch_count() - launches0          # our kernels launched inside the timed region
        if args.dump_outputs and rank == 0:                     # taken before any later call writes the buffer again
            last = gathers[(args.steps - 1) % 2].view(0, world * B) if world > 1 else local_out
            dump = last.index_select(0, torch.from_numpy(dump_clips(world * B)).to(dev))
        # keep the sampler alive for a few more identical steps if the timed region was very short
        t_end = time.time() + 0.25
        while time.time() < t_end and len(clk.samples) < 8:
            pkg.feature_extraction_batch(clips, FS, WINDOW, STEP, deltas=True, out=local_out, plan=plan)
            torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "features.npy"), dump.cpu().numpy())
    ms_per_step = ms_total / args.steps
    frames_per_step = world * B * T
    value = frames_per_step / (ms_per_step * 1e-3)
    scaling_detail = None
    if world > 1:
        timed("none", 3)
        ms_none, _ = timed("none", args.steps)
        timed("nccl", 3)
        ms_nccl, _ = timed("nccl", args.steps)
        timed("p2p_store", 3)
        ms_store, _ = timed("p2p_store", args.steps)
        gather_bytes = (world - 1) * B * 68 * T * 4
        scaling_detail = {"gather": "copy-engine push: every rank's finished block goes into rank 0's peer-mapped buffer (NVLink) on a second stream, "
                                    "under the next step's kernels; all pushes complete inside the timed region",
                          "frames_per_s_with_gather": value,
                          "frames_per_s_without_gather": frames_per_step / (ms_none / args.steps * 1e-3),
                          "frames_per_s_with_nccl_gather": frames_per_step / (ms_nccl / args.steps * 1e-3),
                          "frames_per_s_with_gather_fused_into_kernel_stores": frames_per_step / (ms_store / args.steps * 1e-3),
                          "ms_per_step": {"ce_push_gather": ms_per_step, "no_gather": ms_none / args.steps, "nccl_gather": ms_nccl / args.steps,
                                          "kernel_store_gather": ms_store / args.steps},
                          "root_ingress_bytes_per_step": gather_bytes,
                          "root_ingress_GBps": gather_bytes / (ms_per_step * 1e-3) / 1e9,
                          "limiter": "root NVLink ingress: (N-1) blocks of 108.5 MB per step against ~770 GB/s measured per direction "
                                     "(at N = 8 the gather, not the kernels, sets the step time)"}
        # the gathered tensor on the root holds every rank's block (spot check against the local result)
        timed("ce", 2)
        if rank == 0:
            full = gathers[1].view(0, world * B)
            pkg.feature_extraction_batch(clips, FS, WINDOW, STEP, deltas=True, out=local_out, plan=plan)
            torch.cuda.synchronize()
            assert torch.equal(full[:B], local_out), "gather buffer does not hold rank 0's block"
            assert torch.isfinite(full[(world - 1) * B:]).all() and full[(world - 1) * B:, 1].abs().sum() > 0, "last rank's block missing"

    # ---- end to end through the C ABI host entry point: pinned host clips -> pinned host features
    e2e = None
    if not args.no_e2e:
        pipe = HostPipeline(FS, WINDOW, STEP, CLIP_SAMPLES, max_clips=B, device=local_rank, bind_numa=False)
        pipe.h_in[:] = clips.cpu().numpy()
        host_out = pipe.run()                  # warm-up (allocations, plan)
        for _ in range(2):
            pipe.run()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        n_e2e = max(3, min(args.steps, 10))
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            host_out = pipe.run()
        dt = (time.perf_counter() - t0) / n_e2e
        td = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(td, op=dist.ReduceOp.MAX)
        dt = float(td.item())
        e2e = {"value": frames_per_step / dt, "unit": "frames/s", "h2d_bytes_per_step": int(pipe.h_in.nbytes),
               "d2h_bytes_per_step": int(host_out.nbytes), "ms_per_step": 1e3 * dt,
               "api": "b200aa_st_features_host (C ABI via ctypes; pinned host int16 in, pinned host float32 out; inside: ~32 MB "
                      "chunks, H2D / b200aa_clip_stats + b200aa_st_features / D2H round-robin on three streams)",
               "numa": bound}
        # parity spot check of the e2e result against the device-resident result
        pkg.feature_extraction_batch(clips, FS, WINDOW, STEP, deltas=True, out=local_out, plan=plan)
        torch.cuda.synchronize()
        assert (host_out[:4] == local_out[:4].cpu().numpy()).all(), "host entry point and device path disagree"

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = hbm_peak()
    alg_bytes = B * ALG_BYTES_PER_CLIP
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    nf = ncu_facts()
    inst = nf.get("st_kernel_warp_instructions_per_launch")
    sm_clock_hz = 1e6 * (clk.summary()["sm_mhz"] or 1965)
    issue_frac = (inst / (kernel_ms * 1e-3) / (148 * 4 * sm_clock_hz)) if inst else None
    line = {"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "ours", "config": CONFIG,
            "detail": {"l2": "inputs larger than L2 (320 MB int16 clips + 108 MB output per step vs 126 MB L2); no explicit flush",
                       "kernel_kind": plan.kernel_kind(), "numa": bound,
                       **({"lib_override": os.environ["B200AA_LIB"]} if os.environ.get("B200AA_LIB") else {})},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": nf.get("st_kernel_dram_bytes_per_launch"), "traffic_source": nf.get("source"),
                         "peak_source": peak_src, "kernel": "fused short-term feature kernel",
                         "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": alg_bytes,
                         "binding_bound": "fp32_issue",
                         "fp32_issue_frac": issue_frac, "inst_per_frame": (inst / (B * T)) if inst else None,
                         "issue_slot_utilisation_ncu": nf.get("st_kernel_issue_slot_utilisation"),
                         "note": "the kernel is instruction-issue bound, not HBM bound (DESIGN.md): ~30 kFLOP per 1074 B frame; "
                                 "fp32_issue_frac = warp instructions per launch (ncu capture) / kernel time / (148 SMs x 4 "
                                 "schedulers x SM clock)"},
            "clocks": clk.summary(), "e2e": e2e, "gpu_launches": int(launches)}
    if scaling_detail:
        line["scaling_detail"] = scaling_detail
    if args.dump_outputs:
        line["dump_outputs"] = {"features.npy": {"shape": [DUMP_CLIPS, 68, T], "dtype": "float32",
                                                 "clips": "numpy.random.default_rng(0).choice(%d, %d, replace=False), sorted"
                                                          % (world * B, DUMP_CLIPS)}}
    if world == 1 and not args.no_cpu:
        if full_affinity is not None:
            os.sched_setaffinity(0, full_affinity)       # the CPU baseline uses every core of the box, not only the GPU's node
        line["cpu_baseline"], _, _ = cpu_baseline(target_seconds=30.0)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg (profiling runs)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-pipeline leg (profiling runs under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's features (seeded sample of clips) to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: N independent shards are not possible in one process
        raise SystemExit("--gpus %d needs torchrun (python -m torch.distributed.run --nproc-per-node %d bench.py ...)"
                         % (args.gpus, args.gpus))
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
