#!/usr/bin/env python3
"""Benchmark of the hot path: 1080p CQP I+P H.264 encode, frames/s (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: the whole synthetic clip of the workload
(default: BASELINE.json configs[2], 1920x1088 NV12, 600 frames, GOP 60, QP 25, +-16 full search,
CABAC -- the configuration the metric is quoted on; it fits one GPU) encoded GOP-parallel.
With N > 1 (torchrun, one rank per GPU) every rank encodes its own 600-frame share of a 600*N-frame
clip (GOP g -> rank g % N): closed GOPs share no data, so there is no data-path collective and
the scaling is weak.  `value` = all frames of all ranks / max-over-ranks device time with the clip
already resident in HBM; `e2e` = the same through the C ABI with pinned HOST buffers, H2D of the
raw frames and D2H of the bytestream inside the timed region.

--impl reference times the CPU implementation of the same path (the golden model under oracle/,
the reference itself having no CPU macroblock encoder: its encoder is Allwinner silicon,
kernel/cedar.c:1176) on all host cores, on a bounded sample of the same workload.

--dump-outputs DIR writes what the timed encode returned in its last step (see dump_outputs) for an output-for-output
comparison of two builds: the synthetic clip depends on the arguments only.
"""
import os
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")  # before CUDA initialises: side streams must not share queues
import argparse
import json
import math
import os
import sys
import threading
import time

sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from as it found it (it may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
DUMP_LIMIT = 64 << 20  # bytes that --dump-outputs writes at most

WORKLOADS = {
    # name: (width, height, fmt, frames, gop, qp, me_range, cabac)
    "1080p_nv12_600f_gop60_qp25": (1920, 1088, 0, 600, 60, 25, 16, 1),
    "720p_nv12_300f_gop30_qp25": (1280, 720, 0, 300, 30, 25, 16, 1),
    "1080p_nv16_300f_gop60_qp25": (1920, 1088, 1, 300, 60, 25, 16, 1),
    "2160p_nv12_1200f_gop60_qp25_me64": (3840, 2160, 0, 1200, 60, 25, 64, 1),
    "480p_nv12_30f_gop25_qp24": (854, 480, 0, 30, 25, 24, 16, 1),
}
DEFAULT_WORKLOAD = "1080p_nv12_600f_gop60_qp25"
METRIC = "1080p CQP I+P frames/sec (GOP-parallel)"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ------------------------------------------------------------------------------------------------
# clocks sampling during the timed region (B200_PROFILING.md: clocks line)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.dev = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.dev, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.dev, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.dev)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.05)

    def start(self):
        if self.nv:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join()
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the golden model on the host cores (cpu_baseline leg and --impl reference)
# ------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    (w, h, fmt, gop, qp, me, cabac, first, n) = args
    import hashlib
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    enc = O.Encoder(O.make_config(w, h, qp=qp, gop=gop, cabac=cabac, fmt=fmt, me_range=me))
    frames = [O.synth_frame(w, h, first + i, fmt) for i in range(n)]
    t0 = time.perf_counter()
    out = [enc.encode(y, c) for y, c in frames]
    dt = time.perf_counter() - t0
    enc.close()
    # A fresh encoder writes SPS + PPS in front of its first frame (kernel/cedar.c:1058-1061); inside a stream only
    # frame 0 carries them, so for the comparison with the GPU stream they are dropped from later GOPs.
    if first != 0 and out:
        out[0] = out[0][out[0].index(b"\x00\x00\x00\x01\x65"):]
    blob = b"".join(out)
    return n, dt, len(blob), first, hashlib.sha256(blob).hexdigest()


def cpu_sample(workload, frames_per_core, cores):
    """Every core encodes the first `frames_per_core` frames of a different GOP of the workload.
    Returns (frames/s, frames, wall seconds, [(first frame, frames, bytes, sha256 of those frames' bytes)])."""
    import multiprocessing as mp
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    O.build()
    w, h, fmt, nframes, gop, qp, me, cabac = WORKLOADS[workload]
    jobs = []
    for i in range(cores):
        first = (i * gop) % max(nframes, 1)
        jobs.append((w, h, fmt, gop, qp, me, cabac, first, min(frames_per_core, nframes - first)))
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(cores) as pool:
        res = pool.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    total = sum(r[0] for r in res)
    slowest = max(r[1] for r in res)
    return total / slowest, total, wall, [(r[3], r[0], r[2], r[4]) for r in res]


def parity_block(gops, data, sizes):
    """Golden-model GOPs (cpu_sample) against the same frames cut out of the stream the timed handles produced."""
    import hashlib
    import numpy as np
    offs = np.concatenate([[0], np.cumsum(np.asarray(sizes, dtype=np.int64))])
    seen, bad = set(), []
    for first, n, nbytes, sha in gops:
        if first in seen or first + n > len(sizes):
            continue
        seen.add(first)
        got = bytes(data[int(offs[first]):int(offs[first + n])])
        if len(got) != nbytes or hashlib.sha256(got).hexdigest() != sha:
            bad.append(first)
    return {"gops_checked": len(seen), "frames_checked": sum(n for f, n, _, _ in {g[0]: g for g in gops}.values()),
            "equal": not bad, "mismatching_gops_first_frame": bad,
            "how": "SHA-256 of the golden model's bytes for each sampled GOP == SHA-256 of the same frames of the stream "
                   "downloaded from the timed handle"}


def dump_outputs(out_dir, stream, sizes, suffix=""):
    """--dump-outputs: the Annex-B bytestream of the clip (float32, one value per byte) and the size of every frame in it
    (float64), as .npy files.  A stream beyond DUMP_LIMIT is written as a fixed, seeded sample of its bytes
    (stream_sample) with their positions (stream_sample_index)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    out = {"frame_sizes": np.asarray(sizes, np.float64)}
    room = DUMP_LIMIT - out["frame_sizes"].nbytes - 4096  # 4096: the .npy headers
    if 4 * len(stream) <= room:
        out["stream"] = np.asarray(stream, np.float32)
    else:
        idx = np.unique(np.random.default_rng(0).integers(0, len(stream), room // 12))
        out["stream_sample"] = np.asarray(stream[idx], np.float32)
        out["stream_sample_index"] = idx.astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def run_reference(args, rank, world):
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    w, h, fmt, nframes, gop, qp, me, cabac = WORKLOADS[args.workload]
    fpc = args.cpu_frames
    for _ in range(args.warmup if args.warmup < 1 else 1):
        cpu_sample(args.workload, 1, cores)
    vals, t_all = [], 0.0
    for _ in range(args.steps):
        fps, total, wall, _ = cpu_sample(args.workload, fpc, cores)
        vals.append(fps)
        t_all += wall
    value = sum(vals) / len(vals)
    sample = "%d cores x first %d frames (1 I + %d P) of distinct GOPs of the workload clip" % (cores, fpc, fpc - 1)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_all / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": args.workload, "width": w, "height": h, "frames": nframes, "gop": gop, "qp": qp,
                   "me_range": me, "entropy": "cabac" if cabac else "cavlc", "sample": sample},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "per_core": value / cores, "kind": "port", "sample": sample,
                         "note": "reference has no CPU macroblock encoder (Cedar VE silicon); this is the C golden "
                                 "model of the same algorithm, GOP-parallel across processes"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0



# ------------------------------------------------------------------------------------------------
# Secondary measurements (other BASELINE.json configs, strong scaling): the same timing rules as the headline
# ------------------------------------------------------------------------------------------------
def measure_share(torch, cx, api, synth, spec, frame_ids, local_rank, steps, warmup, nhandles, sync, max_over_ranks,
                  first_frame_index=0, repeat_content=1, noise=False):
    """Encodes this rank's frames of a clip (`frame_ids`, whole GOPs, already in encode order) `steps` times on `nhandles`
    handles.  Returns device-resident and end-to-end milliseconds (max over ranks), per-GOP SHA-256s, stream bytes, SSE.
    repeat_content > 1: the share is `repeat_content` clips of len(frame_ids) frames with the same content (a clip too
    long to keep resident is encoded wave after wave from the same resident frames)."""
    import hashlib
    import threading
    w, h, fmt, _, gop, qp, me, cabac = spec
    n = len(frame_ids)
    if n == 0:  # a rank without work still takes part in the barriers
        sync(), sync()
        ms_dev = max_over_ranks(0.0)
        sync(), sync()
        ms_e2e = max_over_ranks(0.0)
        return {"handles": 0, "frames": 0, "ms_dev": ms_dev, "ms_e2e": ms_e2e, "gop_sha": [], "bytes": 0, "sse": 0.0, "h2d": 0, "d2h": 0}
    cfg = api.make_config(w, h, qp=qp, gop=gop, cabac=cabac, fmt=fmt, me_range=me, device=local_rank, max_clip_frames=n)
    encs = []
    for _ in range(max(1, nhandles)):
        try:
            encs.append(cx.Encoder(cfg))
        except OSError:
            if not encs:
                raise
            break
    staging = torch.from_numpy(encs[0].clip_input(n))
    for i in range(0, n, 20):
        part = synth.synth_clip(w, h, frame_ids[i:i + 20], fmt, device="cuda")
        if noise:  # temporally uncorrelated noise: nothing for the search to find, every macroblock full of coefficients
            gen = torch.Generator(device="cuda").manual_seed(1234 + i)
            part = torch.randint(0, 256, part.shape, dtype=torch.uint8, device="cuda", generator=gen)
        staging[i:i + len(part)].copy_(part)
    torch.cuda.synchronize()
    for e in encs[1:]:
        torch.from_numpy(e.clip_input(n)).copy_(staging[:n])
    strs = [torch.cuda.ExternalStream(e.stream_ptr(), device=torch.device("cuda", local_rank)) for e in encs]

    def run(total_steps, body):
        errs = []

        def work(i):
            try:
                for _ in range(i, total_steps, len(encs)):
                    body(encs[i])
            except Exception as ex:
                errs.append(ex)
        th = [threading.Thread(target=work, args=(i,)) for i in range(len(encs))]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if errs:
            raise errs[0]

    def timed(total_steps, body):
        ev0 = [torch.cuda.Event(enable_timing=True) for _ in strs]
        ev1 = [torch.cuda.Event(enable_timing=True) for _ in strs]
        sync()
        for e, st in zip(ev0, strs):
            e.record(st)
        run(total_steps, body)
        for e, st in zip(ev1, strs):
            e.record(st)
        sync()
        return max_over_ranks(max(a.elapsed_time(b) for a in ev0 for b in ev1))

    def e2e_step(e):
        e.clip_upload(n)
        e.clip_encode(n, first_frame_index)
        e.clip_download(n)
    run(len(encs), e2e_step)  # first: a download makes the library grow its entropy buffers if this content needs it
    run(max(warmup, 1) * len(encs), lambda e: e.clip_encode(n, first_frame_index))
    ms_dev = timed(steps * repeat_content, lambda e: e.clip_encode(n, first_frame_index))
    run(len(encs), e2e_step)
    ms_e2e = timed(steps * repeat_content, e2e_step)
    data, sizes = encs[0].clip_download(n)
    data = data.tobytes()
    sse = float(encs[0].sse_y(n).sum())
    shas, off = [], 0
    for g0 in range(0, n, gop):
        nb = int(sizes[g0:g0 + gop].sum())
        shas.append((int(frame_ids[g0]), hashlib.sha256(data[off:off + nb]).hexdigest()))
        off += nb
    fb = encs[0].frame_bytes
    for e in encs:
        e.close()
    return {"frames": n, "ms_dev": ms_dev, "ms_e2e": ms_e2e, "gop_sha": shas, "bytes": len(data), "sse": sse,
            "h2d": n * fb, "d2h": len(data) + 4 * n + 16, "handles": len(encs)}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_gpu(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    import cedarx_h264_encoder_b200 as cx
    from cedarx_h264_encoder_b200 import api, partition, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the encoder has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    w, h, fmt, nframes, gop, qp, me, cabac = WORKLOADS[args.workload]
    total_frames = nframes * world
    my_frames = partition.frames_for_rank(total_frames, gop, rank, world)
    n = len(my_frames)
    # Where this rank's share starts in the stream: only the rank that owns stream frame 0 emits SPS + PPS
    # (kernel/cedar.c:1058-1061), so that the rank streams concatenate GOP by GOP into the single stream.
    ffi = my_frames[0] if my_frames else 0

    cfg = api.make_config(w, h, qp=qp, gop=gop, cabac=cabac, fmt=fmt, me_range=me, device=local_rank,
                          max_clip_frames=n, gops_in_flight=args.lanes, slice_rows=args.slice_rows)
    enc = cx.Encoder(cfg)
    stream = torch.cuda.ExternalStream(enc.stream_ptr(), device=torch.device("cuda", local_rank))

    # synthetic clip: generated on the GPU (plumbing), staged into the library's pinned host buffer
    staging = torch.from_numpy(enc.clip_input(n))
    chunk = 20
    for i in range(0, n, chunk):
        part = synth.synth_clip(w, h, my_frames[i:i + chunk], fmt, device="cuda")
        staging[i:i + len(part)].copy_(part)
    torch.cuda.synchronize()
    # A handle is one latency-bound chain of dependent launches (60 lock-step passes per GOP); a second handle on the
    # same GPU, driven from its own host thread, fills the SMs the first one leaves idle.  Steps alternate between them.
    # 0 = two or three, whichever leaves the shorter tail for this number of steps (measured: two clips in flight take
    # 1.55x and three 2.24x the time of one; rounds of the round-robin schedule with fewer busy handles cost accordingly)
    def schedule_cost(c, k):
        rel = {0: 0.0, 1: 1.0, 2: 1.55, 3: 2.24}
        return sum(rel[min(c, k - r * c)] for r in range(-(-k // c)))
    nhandles = args.clips_in_flight or min((2, 3), key=lambda c: schedule_cost(c, max(args.steps, 1)))
    encs, streams = [enc], [stream]
    for _ in range(max(nhandles, 1) - 1):
        try:
            e = cx.Encoder(cfg)
        except OSError as ex:  # a 4K 1200-frame clip is 15 GB of device and of pinned host memory per handle
            print("bench.py: no memory for handle %d (%s); continuing with %d" % (len(encs) + 1, ex, len(encs)), file=sys.stderr)
            break
        torch.from_numpy(e.clip_input(n)).copy_(staging[:n])
        encs.append(e)
        streams.append(torch.cuda.ExternalStream(e.stream_ptr(), device=torch.device("cuda", local_rank)))

    def run_steps(handles, steps, body):
        """steps passes of body(handle), round robin over the handles, one host thread per handle."""
        import threading
        errs = []

        def work(i):
            try:
                for _ in range(i, steps, len(handles)):
                    body(handles[i])
            except Exception as ex:  # surfaced below: a failed step must fail the bench
                errs.append(ex)
        if len(handles) == 1:
            work(0)
        else:
            th = [threading.Thread(target=work, args=(i,)) for i in range(len(handles))]
            for t in th:
                t.start()
            for t in th:
                t.join()
        if errs:
            raise errs[0]

    def timed(handles, strs, steps, body):
        """Device time of `steps` passes: CUDA events on every handle's launching stream, earliest start to latest end."""
        ev0 = [torch.cuda.Event(enable_timing=True) for _ in strs]
        ev1 = [torch.cuda.Event(enable_timing=True) for _ in strs]
        barrier()
        for e, st in zip(ev0, strs):
            e.record(st)
        run_steps(handles, steps, body)
        for e, st in zip(ev1, strs):
            e.record(st)
        barrier()
        return max_over_ranks(max(a.elapsed_time(b) for a in ev0 for b in ev1))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # -------- device-resident throughput (`value`) --------
    for e in encs:
        e.clip_upload(n)
        e.clip_encode(n, ffi)
        e.clip_download(n)  # grows the entropy buffers now if this content needs it: the timed encodes must not overflow
    run_steps(encs, max(args.warmup, 0) * len(encs), lambda e: e.clip_encode(n, ffi))
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = sum(e.launch_count() for e in encs)
    ms_dev = timed(encs, streams, args.steps, lambda e: e.clip_encode(n, ffi))
    clocks = sampler.stop()
    launches = sum(e.launch_count() for e in encs) - launches0
    # the same steps through one handle alone (one clip in flight): the latency-bound figure
    ms_single = timed(encs[:1], streams[:1], args.steps, lambda e: e.clip_encode(n, ffi)) if len(encs) > 1 else ms_dev
    data, sizes = enc.clip_download(n)
    data = data.copy()  # the view is only valid until the next clip call on this handle
    stream_bytes = int(len(data))
    import hashlib
    stream_sha = hashlib.sha256(data.tobytes()).hexdigest()
    # every handle encoded the same clip in the timed region: their streams must be the same bytes
    handles_identical = all(hashlib.sha256(e.clip_download(n)[0].tobytes()).hexdigest() == stream_sha for e in encs[1:])
    sse = enc.sse_y(n)
    # CABAC bins of the clip (debug read 6: one count per slice NAL), for the per-bin cost of the two coder kernels
    import numpy as np
    nbins, nsl, bins_p_frame = 0, 1, 0.0
    if cabac:
        mbh_ = (h + 15) // 16
        nsl = 1 if not args.slice_rows or args.slice_rows >= mbh_ else -(-mbh_ // args.slice_rows)
        bins = np.zeros(n * nsl, np.uint32)
        enc.L.cedar_b200_debug_read(enc.h, 6, bins.ctypes.data, bins.nbytes)
        nbins = int(bins.sum())
        per_frame_bins = bins.reshape(n, nsl).sum(axis=1)
        p_mask = (np.arange(n) % gop) != 0
        bins_p_frame = float(per_frame_bins[p_mask].mean()) if p_mask.any() else 0.0

    # -------- end to end through the C ABI with host buffers (`e2e`) --------
    def e2e_step(e):
        e.clip_upload(n)
        e.clip_encode(n, ffi)
        e.clip_download(n)
    run_steps(encs, min(args.warmup, 1) * len(encs), e2e_step)
    ms_e2e = timed(encs, streams, args.steps, e2e_step)

    # -------- per-kernel device times with CUDA events on the launching stream --------
    # live: inside the overlapped multi-stream run (what the timed region looks like);
    # standalone: the same clip with every kernel issued on one stream (what ncu would see).
    enc.profile_enable(1)
    enc.profile_read(reset=True)
    enc.clip_encode(n, ffi)
    prof_live = enc.profile_read(reset=True)
    enc.profile_enable(2)
    enc.clip_encode(n, ffi)
    prof = enc.profile_read(reset=True)
    # measurement builds of the kernels (same bytes, work counters): executed VABSDIFF4 lane-instructions of the pruned
    # search and the CABAC bins per context (for the serial-chain bound of cabac_resolve_kernel)
    enc.profile_enable(3)
    enc.profile_read(reset=True)
    enc.clip_encode(n, ffi)
    counters = np.zeros(520, np.uint64)
    enc.L.cedar_b200_debug_read(enc.h, 8, counters.ctypes.data, counters.nbytes)
    enc.profile_read(reset=True)
    enc.profile_enable(0)
    torch.cuda.synchronize()
    me_executed = int(counters[0])
    ctx_bins = counters[8:8 + 460].astype(np.int64)
    extra_meas = {}
    if rank == 0 and world == 1 and not args.no_extras:
        # (a) the same clip with the pruning of the motion search switched off (content that defeats it pays this)
        os.environ["CEDAR_B200_NO_PRUNE"] = "1"
        e_np = cx.Encoder(cfg)
        del os.environ["CEDAR_B200_NO_PRUNE"]
        torch.from_numpy(e_np.clip_input(n)).copy_(staging[:n])
        e_np.clip_upload(n)
        e_np.profile_enable(3)
        e_np.clip_encode(n, ffi)
        e_np.profile_read(reset=True)
        e_np.clip_encode(n, ffi)
        cnt_np = np.zeros(520, np.uint64)
        e_np.L.cedar_b200_debug_read(e_np.h, 8, cnt_np.ctypes.data, cnt_np.nbytes)
        p_np = e_np.profile_read(reset=True)
        d_np, _ = e_np.clip_download(n)
        extra_meas["no_prune"] = {"me_kernel_ms": p_np.get("me_kernel", (0.0, 0))[0], "executed": int(cnt_np[0]),
                                  "same_bytes": hashlib.sha256(d_np.tobytes()).hexdigest() == stream_sha}
        e_np.close()
        # (b) the dependent chain of ONE macroblock through deblock_kernel: a picture one macroblock row high has no
        # vertical dependencies, so its launch time / macroblocks = what one warp needs per macroblock with nothing to wait for
        e_row = cx.Encoder(api.make_config(w, 16, qp=qp, gop=2, cabac=cabac, fmt=fmt, me_range=me, device=local_rank,
                                           max_clip_frames=2, gops_in_flight=1))
        torch.from_numpy(e_row.clip_input(2)).copy_(synth.synth_clip(w, 16, [0, 1], fmt, device="cuda").cpu())
        e_row.clip_upload(2)
        e_row.clip_encode(2, 0)
        e_row.profile_enable(2)
        e_row.profile_read(reset=True)
        for _ in range(5):
            e_row.clip_encode(2, 0)
        p_row = e_row.profile_read(reset=True)
        e_row.close()
        if "deblock_kernel" in p_row:
            extra_meas["deblock_row_ms_per_launch"] = p_row["deblock_kernel"][0] / p_row["deblock_kernel"][1]

    value = total_frames * args.steps / (ms_dev * 1e-3)
    e2e = total_frames * args.steps / (ms_e2e * 1e-3)

    # -------- slice-parallel entropy coding (north star: MB rows per slice configurable, bitrate cost reported) -----
    # Same clip, same settings, slice_rows = N: every N macroblock rows are their own slice NAL and get their own
    # serial coder.  Not the headline (the reference writes one slice per picture, cedar.c:992-993).
    slice_report = None
    if world == 1 and not args.no_slice_report and args.slice_rows == 0:
        slice_report = []
        mbh = (h + 15) // 16
        for rows in sorted({(mbh + 3) // 4, (mbh + 15) // 16}, reverse=True):
            cfg2 = api.make_config(w, h, qp=qp, gop=gop, cabac=cabac, fmt=fmt, me_range=me, device=local_rank,
                                   max_clip_frames=n, gops_in_flight=args.lanes, slice_rows=rows)
            enc2 = cx.Encoder(cfg2)
            torch.from_numpy(enc2.clip_input(n)).copy_(staging[:n])
            enc2.clip_upload(n)
            st2 = torch.cuda.ExternalStream(enc2.stream_ptr(), device=torch.device("cuda", local_rank))
            for _ in range(2):
                enc2.clip_encode(n, 0)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st2)
            for _ in range(args.steps):
                enc2.clip_encode(n, 0)
            b.record(st2)
            torch.cuda.synchronize()
            d2, _ = enc2.clip_download(n)
            sse2 = enc2.sse_y(n)
            slice_report.append({"slice_rows": rows, "slices_per_picture": -(-mbh // rows),
                                 "value": n * args.steps / (a.elapsed_time(b) * 1e-3), "unit": "frames/s",
                                 "kbit_per_frame": round(len(d2) * 8 / 1000.0 / n, 2),
                                 "bitrate_cost_pct": round(100.0 * (len(d2) - stream_bytes) / stream_bytes, 3),
                                 "y_psnr_delta_db": round(10 * math.log10(float(sse.sum()) / float(sse2.sum())), 4)})
            enc2.close()
    parity_ok = handles_identical
    parity_extra_ok = True
    # -------- GOP-parallel merge check on hardware (SURVEY 8e invariant, BASELINE.md gate 4) --------
    # Every rank hashes each closed GOP of the stream its timed handle produced; rank 0 gathers them, checks that every
    # GOP of the N x 600-frame clip is there exactly once, and re-encodes spot GOPs owned by OTHER ranks on its own GPU
    # (with their first_frame_index): same bytes => the rank streams concatenate to the stream one GPU produces.
    my_gops = partition.gops_for_rank(total_frames, gop, rank, world)
    offs = np.concatenate([[0], np.cumsum(sizes.astype(np.int64))])
    gop_sha = {}
    for i, g in enumerate(my_gops):
        nf = len(partition.frames_of_gop(total_frames, gop, g))
        gop_sha[g] = hashlib.sha256(data[int(offs[i * gop]):int(offs[i * gop + nf])].tobytes()).hexdigest()
    merged = None
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, gop_sha)
        if rank == 0:
            allg = {}
            for d in gathered:
                allg.update(d)
            spots = [g for g in (1, partition.num_gops(total_frames, gop) - 1) if g % world != 0]
            spot_ok = []
            for g in spots:
                ids = partition.frames_of_gop(total_frames, gop, g)
                staging[:len(ids)].copy_(synth.synth_clip(w, h, ids, fmt, device="cuda"))
                torch.cuda.synchronize()
                enc.clip_upload(len(ids))
                enc.clip_encode(len(ids), g * gop)
                d2, _ = enc.clip_download(len(ids))
                spot_ok.append(hashlib.sha256(d2.tobytes()).hexdigest() == allg.get(g))
            merged = {"gops_total": partition.num_gops(total_frames, gop), "gops_gathered": len(allg),
                      "spot_gops_reencoded_on_rank0": spots, "merged_equal": bool(spot_ok) and all(spot_ok) and
                      len(allg) == partition.num_gops(total_frames, gop),
                      "how": "per-GOP SHA-256 all_gather; rank 0 re-encodes GOPs owned by other ranks with their "
                             "first_frame_index and compares"}
            parity_extra_ok = merged["merged_equal"]
        dist.barrier()

    # -------- the other BASELINE.json configs and strong scaling (same timing rules, fewer steps) --------
    def sync_all():
        barrier()
    others, strong = None, None
    if not args.no_extras:
        st_ = max(2, min(args.steps, 3))
        others = {}
        if world == 1:
            plan = [("720p_nv12_300f_gop30_qp25", 300), ("1080p_nv16_300f_gop60_qp25", 300),
                    ("2160p_nv12_1200f_gop60_qp25_me64", 120)]
        else:
            plan = []
        for name, nfr in plan:
            spec = WORKLOADS[name]
            r_ = measure_share(torch, cx, api, synth, spec, list(range(nfr)), local_rank, st_, 1, 2, sync_all, max_over_ranks)
            W16_, H16_ = ((spec[0] + 15) // 16) * 16, ((spec[1] + 15) // 16) * 16
            mse_ = r_["sse"] / (nfr * W16_ * H16_)
            others[name] = {"frames_encoded": nfr, "value": nfr * st_ / (r_["ms_dev"] * 1e-3), "unit": "frames/s",
                            "e2e": nfr * st_ / (r_["ms_e2e"] * 1e-3), "handles": r_["handles"],
                            "kbit_per_frame": round(r_["bytes"] * 8 / 1000.0 / nfr, 2),
                            "y_psnr_db": round(10 * math.log10(255.0 ** 2 / mse_), 3) if mse_ > 0 else None,
                            "stream_sha256": hashlib.sha256(repr(r_["gop_sha"]).encode()).hexdigest()[:16]}
        # worst-case content: white noise (the exact pruning of the search cannot skip anything, the entropy coder sees
        # ~20 x the bins; the entropy buffers grow on the first encode, which is part of the warm-up)
        if world == 1:
            try:
                spec = WORKLOADS[DEFAULT_WORKLOAD]
                r_ = measure_share(torch, cx, api, synth, spec, list(range(120)), local_rank, 2, 1, 2, sync_all, max_over_ranks, noise=True)
                others["1080p_white_noise_120f"] = {"frames_encoded": 120, "value": 120 * 2 / (r_["ms_dev"] * 1e-3), "unit": "frames/s",
                                                    "e2e": 120 * 2 / (r_["ms_e2e"] * 1e-3), "handles": r_["handles"],
                                                    "kbit_per_frame": round(r_["bytes"] * 8 / 1000.0 / 120, 2),
                                                    "note": "uncorrelated noise at QP 25: content that defeats the search's pruning "
                                                            "and fills every macroblock with coefficients"}
            except Exception as ex:  # reported, not fatal: the headline workload is the contract
                others["1080p_white_noise_120f"] = {"error": str(ex)}
        # strong scaling: a FIXED clip split GOP g -> rank g % N (BASELINE.md 3: 960 frames = 16 GOPs for a clean 8x;
        # 4800 frames = 80 GOPs so that 8 ranks still hold 10 GOPs each; config 5 = 4K, 1200 frames, +-64)
        strong = {}
        dspec = WORKLOADS[DEFAULT_WORKLOAD]
        for label, spec, clip_frames, max_res_gops in (("1080p_960f", dspec, 960, 16), ("1080p_4800f", dspec, 4800, 10),
                                                       ("2160p_1200f_me64", WORKLOADS["2160p_nv12_1200f_gop60_qp25_me64"], 1200, 5)):
            g_ = spec[4]
            share = partition.frames_for_rank(clip_frames, g_, rank, world)
            share_gops = len(share) // g_
            res_gops = min(share_gops, max_res_gops)
            rep = -(-share_gops // res_gops) if res_gops else 1
            if world > 1:  # every rank must run the same number of timed passes
                t_ = torch.tensor([rep], device="cuda")
                dist.all_reduce(t_, op=dist.ReduceOp.MAX)
                rep = int(t_.item())
            r_ = measure_share(torch, cx, api, synth, spec, share[:res_gops * g_], local_rank, st_, 1, 2, sync_all, max_over_ranks,
                               first_frame_index=0, repeat_content=rep)
            strong[label] = {"clip_frames": clip_frames, "gops": clip_frames // g_, "value": clip_frames * st_ / (r_["ms_dev"] * 1e-3),
                             "e2e": clip_frames * st_ / (r_["ms_e2e"] * 1e-3), "unit": "frames/s",
                             "frames_resident_rank0": res_gops * g_, "passes_per_step": rep,
                             "ceiling_speedup": partition.scaling_ceiling(clip_frames, g_, world)}
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        # roofline denominator of me_kernel: the issue rate of VABSDIFF4.U8.ACC, measured LIVE on this GPU with the
        # micro-benchmark tools/vabsdiff_bench (built by __graft_entry__.build()); else the committed measurement
        simd_peak, simd_src = 18.54e12, "profiles/vabsdiff4_peak.json (round 1 measurement on this pool)"
        try:
            simd_peak = float(json.load(open(os.path.join(ROOT, "profiles", "vabsdiff4_peak.json")))["vabsdiff4_lane_instr_per_s"])
        except Exception:
            pass
        try:
            import subprocess
            out = subprocess.run([os.path.join(ROOT, "tools", "vabsdiff_bench")], capture_output=True, text=True, timeout=60,
                                 env=dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local_rank))))
            live = json.loads(out.stdout.strip().splitlines()[-1])
            simd_peak = float(live["vabsdiff4_lane_instr_per_s"])
            simd_src = "measured live on this GPU by tools/vabsdiff_bench (%.1f lane-instr/SM/clk)" % live["per_sm_per_clk_at_max_clock"]
        except Exception:
            pass
        nmb = (((w + 15) // 16) * ((h + 15) // 16))
        W16, H16 = ((w + 15) // 16) * 16, ((h + 15) // 16) * 16
        kernels = {}
        tot_ms = sum(v[0] for v in prof.values()) or 1.0
        for name, (ms, cnt) in prof.items():
            kernels[name] = {"ms_total": round(ms, 4), "launches": cnt, "share": round(ms / tot_ms, 4),
                             "ms_total_live": round(prof_live.get(name, (0.0, 0))[0], 4)}
        for name, (ms, cnt) in prof_live.items():  # launches that only exist in the overlapped schedule (fused kernels)
            if name not in kernels:
                kernels[name] = {"ms_total": None, "launches": cnt, "share": None, "ms_total_live": round(ms, 4)}
        dominant = max(prof.items(), key=lambda kv: kv[1][0])[0] if prof else None
        clk_hz = (clocks.get("sm_mhz") or 1965) * 1e6
        my_gops_n = len(partition.gops_for_rank(total_frames, gop, rank, world))
        p_frames = n - my_gops_n
        lanes_ = int(enc.cfg.gops_in_flight) or min(16, -(-n // gop))
        rooflines = {}
        if "me_kernel" in prof:
            ms, cnt = prof["me_kernel"]
            instr = p_frames * nmb * (2 * me + 1) ** 2 * 64.0  # algorithmic VABSDIFF4 lane-instructions
            ach = instr / (ms * 1e-3)
            npn = extra_meas.get("no_prune")
            rooflines["me_kernel"] = {
                "kernel": "me_kernel", "bound": "int-simd (VABSDIFF4 issue rate; neither hbm nor tensor)",
                "achieved": ach / 1e12, "peak": simd_peak / 1e12, "unit": "T VABSDIFF4 lane-instr/s", "frac": ach / simd_peak,
                "frac_algorithmic": ach / simd_peak,
                "frac_executed": (me_executed / (ms * 1e-3)) / simd_peak if me_executed else None,
                "executed_over_algorithmic": me_executed / instr if me_executed else None,
                "no_prune": None if not npn else {"ms_per_clip": round(npn["me_kernel_ms"], 3), "frac": (npn["executed"] / (npn["me_kernel_ms"] * 1e-3)) / simd_peak
                                                  if npn["me_kernel_ms"] else None, "executed_over_algorithmic": npn["executed"] / instr,
                                                  "same_bytes": npn["same_bytes"],
                                                  "note": "measurement build (counter + 71 registers): an upper bound of the product kernel's time without pruning"},
                "traffic": {"dram_bytes_per_launch": 43.54e6, "algorithmic_bytes_per_launch": 2.0 * W16 * H16 * 10,
                            "source": "dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of this kernel "
                                      "with the final code (profiles/r02_ncu_me_inter_full_summary.json; 1080p, 10 GOPs in "
                                      "flight, second inter step)"} if args.workload == DEFAULT_WORKLOAD and world == 1 else None,
                "peak_source": simd_src,
                "algorithmic_per_launch": instr / cnt, "avg_launch_ms": ms / cnt,
                "frac_live": instr / (prof_live["me_kernel"][0] * 1e-3) / simd_peak if "me_kernel" in prof_live else None,
                "timing": "CUDA events per launch; frac = standalone (single stream), frac_live = inside the overlapped step",
                "note": "frac / frac_algorithmic count the instructions of the exhaustive search; frac_executed counts what the "
                        "exactly pruned search really issued (counter in the measurement build of the same kernel)"}
        if "deblock_kernel" in prof:
            ms, cnt = prof["deblock_kernel"]
            mbw_, mbh_ = W16 // 16, H16 // 16
            steps = mbw_ + mbh_ - 1  # 1:1 wavefront: macroblock (x, y) after (x - 1, y) and (x, y - 1)
            row = extra_meas.get("deblock_row_ms_per_launch")
            per_mb = row / mbw_ if row else None
            # lower bound of a wavefront step: the luma warp's instructions for one macroblock at one instruction per
            # clock (ncu, profiles/r02_ncu_full_summary.json: 81.3 M warp instructions per launch of 81 600 macroblocks
            # = 1 000 per macroblock for the luma and the chroma warp together, about 600 of them luma)
            floor_ms = steps * 600.0 / clk_hz * 1e3
            rooflines["deblock_kernel"] = {
                "kernel": "deblock_kernel", "bound": "dependency latency (raster-order wavefront)", "unit": "ms per launch",
                "achieved": ms / cnt, "peak": floor_ms, "floor": floor_ms, "frac": floor_ms / (ms / cnt), "traffic": None,
                "wavefront_steps": steps, "cycles_per_step": (ms / cnt) * 1e-3 * clk_hz / steps,
                "one_warp_alone_cycles_per_macroblock": per_mb * 1e-3 * clk_hz if per_mb else None,
                "floor_source": "wavefront steps (mbw + mbh - 1) x the luma warp's ~600 instructions per macroblock at one per "
                                "clock; one_warp_alone = the same kernel on a picture one macroblock row high (nothing to wait "
                                "for, nothing overlapped) / macroblocks",
                "hbm_frac": (2 * W16 * H16 * 1.5 * n / (ms * 1e-3) / 1e9) / hbm_peak}
        if "cabac_resolve_kernel" in prof and ctx_bins.sum() > 0:
            ms, cnt = prof["cabac_resolve_kernel"]
            hot = int(ctx_bins.max())
            chain = 39.0  # cycles per look-up of four bins: LDS 29 (B300_MICROARCH.md) + two dependent ALU operations
            floor_ms = (hot / float(lanes_ * nsl)) / 4.0 * chain / clk_hz * 1e3  # the lanes' slices are coded side by side
            rooflines["cabac_resolve_kernel"] = {
                "kernel": "cabac_resolve_kernel", "bound": "serial chain along the hottest context", "unit": "ms per clip (sum of launches)",
                "achieved": ms, "peak": floor_ms, "floor": floor_ms, "frac": floor_ms / ms, "traffic": None,
                "hottest_context": int(ctx_bins.argmax()), "hottest_context_share": hot / float(ctx_bins.sum()),
                "chain_cycles_per_4_bins": chain,
                "floor_source": "bins of the hottest context per slice (counted by the measurement build) / 4 bins per look-up "
                                "x dependent look-up latency; the sort passes around the chain are the rest",
                "note": "summed over launches that run on side streams, 10 CTAs each: it is not on the reconstruction chain and "
                        "may exceed ms_per_step"}
        if "cabac_code_kernel" in prof and nbins:
            ms, cnt = prof["cabac_code_kernel"]
            ach = ms * 1e-3 * clk_hz / (nbins / float(lanes_ * nsl))
            ipb = None
            try:  # warp instructions per bin from the ncu capture of an inter step (10 slices in one launch)
                cap = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_full_summary.json")))
                for rec in (cap if isinstance(cap, list) else cap.get("launches", [])):
                    if "cabac_code_kernel" in rec.get("kernel", "") and bins_p_frame:
                        ipb = float(rec["smsp__inst_executed.sum"]) / (10 * bins_p_frame)
            except Exception:
                pass
            floor = ipb / 4.0 if ipb else None  # four schedulers, one warp instruction per clock each
            rooflines["cabac_code_kernel"] = {
                "kernel": "cabac_code_kernel", "bound": "instruction issue of one SM (one CTA per slice, all bins in parallel)",
                "unit": "cycles per bin", "achieved": ach, "peak": floor, "floor": floor, "frac": floor / ach if floor else None,
                "traffic": None, "warp_instructions_per_bin": ipb,
                "floor_source": "executed warp instructions per bin (ncu, profiles/r02_ncu_full_summary.json) / 4 issue slots per "
                                "clock of the one SM a slice's coder runs on",
                "note": "summed over launches on side streams (10 CTAs each): not on the reconstruction chain, may exceed ms_per_step"}
        for k, v in rooflines.items():
            v["share_of_summed_kernel_time"] = kernels[k]["share"]
        # Which kernel dominates?  Summed launch durations overstate the CABAC kernels: their launches are 10 CTAs on 10 of
        # the 148 SMs, on side streams beside the chain.  The resource that binds the headline (three chains sharing the
        # GPU) is SM time / instruction issue, so dominance is weighed by duration x SMs the launch occupies; `rooflines`
        # carries the bound of every one of the four either way.
        mbh__ = H16 // 16
        sms = {"cabac_resolve_kernel": min(148, lanes_ * nsl), "cabac_code_kernel": min(148, lanes_ * nsl),
               "deblock_kernel": min(148, -(-mbh__ // 16) * lanes_ * 2), "intra_kernel": min(148, -(-mbh__ // 8) * lanes_)}
        sm_time = {k: v["ms_total"] * sms.get(k, 148) for k, v in kernels.items() if v["ms_total"]}
        tot_sm = sum(sm_time.values()) or 1.0
        for k, v in rooflines.items():
            v["sms_occupied"] = sms.get(k, 148)
            v["share_of_sm_time"] = round(sm_time.get(k, 0.0) / tot_sm, 4)
        by_sm = max(rooflines, key=lambda k: sm_time.get(k, 0.0)) if rooflines else None
        roofline = dict(rooflines[by_sm]) if by_sm else None
        if roofline:
            roofline["dominance"] = {"by_sm_time": by_sm, "by_summed_launch_duration": dominant,
                                     "sm_time_share": {k: round(sm_time[k] / tot_sm, 4) for k in sorted(sm_time, key=sm_time.get, reverse=True)[:5]},
                                     "note": "duration x SMs a launch occupies; the CABAC kernels' launches are 10 CTAs on side "
                                             "streams, off the reconstruction chain; ncu (profiles/): me_kernel executes 50 % of a "
                                             "clip's warp instructions"}
            roofline["on_critical_chain"] = roofline["kernel"] in ("me_kernel", "deblock_kernel")
        hbm = {}
        frame_bytes = W16 * H16 * 3 // 2
        alg = {"inter_kernel": 3 * frame_bytes, "deblock_kernel": 2 * frame_bytes, "ingest_kernel": 2 * frame_bytes,
               "intra_kernel": 2 * frame_bytes, "sse_kernel": 2 * W16 * H16}
        for name, per_frame in alg.items():
            if name in prof:
                ms, cnt = prof[name]
                nfr = {"inter_kernel": n - len(partition.gops_for_rank(total_frames, gop, rank, world)),
                       "intra_kernel": len(partition.gops_for_rank(total_frames, gop, rank, world))}.get(name, n)
                gbs = per_frame * nfr / (ms * 1e-3) / 1e9
                hbm[name] = {"bound": "hbm", "achieved": round(gbs, 2), "peak": hbm_peak, "unit": "GB/s",
                             "frac": round(gbs / hbm_peak, 5), "traffic": None, "peak_source": hbm_src}
        mse = float(sse.sum()) / (n * W16 * H16)
        cabac_stats = None
        if nbins and clocks and clocks.get("sm_mhz"):
            lanes = int(enc.cfg.gops_in_flight) or min(16, -(-n // gop))  # CTAs of a launch = lanes x slices, side by side
            per_cta_bins = nbins / float(lanes * nsl)
            cabac_stats = {"bins_per_clip": nbins, "bins_per_frame": round(nbins / n, 1),
                           "note": "one CTA per slice NAL; cycles per bin = summed launch time x SM clock / bins one CTA codes per "
                                   "clip; resolve is serial along one context's bins, code is parallel over all bins"}
            for k in ("cabac_resolve_kernel", "cabac_code_kernel"):
                if k in prof:
                    cabac_stats[k + "_cycles_per_bin"] = round(prof[k][0] * 1e-3 * clocks["sm_mhz"] * 1e6 / per_cta_bins, 2)
        # host-link ceiling of the end-to-end figure: pinned H2D of every rank's raw clip at once, nothing else running,
        # measured on this pool's 8-GPU box with tools/h2d_peak.py (profiles/r02_h2d_peak.jsonl)
        host_link = None
        try:
            for ln in open(os.path.join(ROOT, "profiles", "r02_h2d_peak.jsonl")):
                rec = json.loads(ln)
                if rec.get("n_gpus") == world:
                    gbps = max(rec["aggregate_GBps"].values())
                    ceil_fps = gbps * 1e9 / enc.frame_bytes
                    host_link = {"aggregate_h2d_GBps": gbps, "frames_per_s_ceiling": round(ceil_fps, 1),
                                 "e2e_frac_of_ceiling": round(e2e / ceil_fps, 4),
                                 "source": "profiles/r02_h2d_peak.jsonl (tools/h2d_peak.py, %d ranks, one NUMA node, 32 host cores)" % world}
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": args.workload, "width": w, "height": h, "format": "nv16" if fmt else "nv12",
                       "frames_per_gpu": n, "gop": gop, "qp": qp, "me_range": me, "entropy": "cabac" if cabac else "cavlc",
                       "slice_rows": args.slice_rows or "one slice per picture (reference layout)",
                       "gops_in_flight": int(enc.cfg.gops_in_flight) or "auto", "parallelism": "gop-parallel x%d" % world,
                       "clips_in_flight": len(encs),
                       "l2": "inputs larger than L2 (%.0f MB raw clip per GPU vs 126 MB)" % (n * enc.frame_bytes / 1e6),
                       "scaling_ceiling_strong": partition.scaling_ceiling(nframes, gop, world)},
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": int(n * enc.frame_bytes) * world,
                    "d2h_bytes_per_step": (stream_bytes + 4 * n + 16) * world, "ms_per_step": ms_e2e / args.steps,
                    "host_link": host_link},
            "gpu_launches": int(launches),
            "one_clip_in_flight": {"value": total_frames * args.steps / (ms_single * 1e-3), "unit": "frames/s",
                                   "ms_per_step": ms_single / args.steps,
                                   "note": "the same steps through a single handle; `kernels`, `roofline` and `slice_parallel` "
                                           "are measured this way"},
            "roofline": roofline,
            "rooflines": rooflines,
            "roofline_hbm_kernels": hbm,
            "kernels": kernels,
            "slice_parallel": slice_report,
            "cabac": cabac_stats,
            "merged": merged,
            "other_workloads": others,
            "strong_scaling": strong,
            "quality": {"y_psnr_db": round(10 * math.log10(255.0 ** 2 / mse), 3) if mse > 0 else None,
                        "kbit_per_frame": round(stream_bytes * 8 / 1000.0 / n, 2)},
        }
        if not args.no_cpu_baseline and world == 1:
            cores = os.cpu_count() or 1
            fps, total, wall, gops = cpu_sample(args.workload, args.cpu_frames, cores)
            line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": cores, "per_core": fps / cores, "kind": "port",
                                    "sample": "%d cores x first %d frames of distinct GOPs (%.1f s wall)" % (
                                        cores, args.cpu_frames, wall)}
            line["parity"] = parity_block(gops, data, sizes)
            line["parity"]["handles_identical"] = handles_identical
            parity_ok = parity_ok and line["parity"]["equal"]
        else:
            line["cpu_baseline"] = None
        print(json.dumps(line))
    if args.dump_outputs:  # `data`: handle 0's stream after its last timed step (every handle's is the same bytes)
        dump_outputs(args.dump_outputs, data, sizes, "_rank%d" % rank if world > 1 else "")
    for e in encs:
        e.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    parity_ok = parity_ok and parity_extra_ok
    if not parity_ok:
        print("bench.py: PARITY FAILURE -- the timed stream differs from the golden model (see \"parity\")", file=sys.stderr)
        return 3
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--lanes", type=int, default=0, help="GOPs in flight per GPU (0 = auto)")
    ap.add_argument("--cpu-frames", type=int, default=60, help="frames per core in the CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--slice-rows", type=int, default=0, help="macroblock rows per slice (0 = one slice per picture)")
    ap.add_argument("--no-slice-report", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the other BASELINE configs and the strong-scaling clips")
    ap.add_argument("--clips-in-flight", type=int, default=0,
                    help="encoder handles per GPU, each on its own host thread; steps alternate between them (0 = 2 or 3, by --steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the stream the timed encode returned in its last step to DIR/*.npy (b200 arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: only the b200 arm returns a whole stream")
    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    if args.impl == "reference":
        return run_reference(args, rank, world)
    return run_gpu(args, rank, local_rank, world)


if __name__ == "__main__":
    sys.exit(main())
