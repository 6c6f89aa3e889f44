#!/usr/bin/env python
"""bench.py -- headline benchmark: spectrogram Msamples/s (cf32, 1024-pt FFT) on N B200s.

Workload (BASELINE.json configs[0] parameters at the roofline-capable size SURVEY.md 8d names):
cf32_le synthetic recording, 2^28 complex samples PER GPU (2 GiB in, 2 GiB of float32 dB out),
1024-point Hann window, 50 % overlap (hop 512), 20*log10(|X|+1e-10), fft-shifted rows.
A "step" is one pass of the whole hot path (decode -> frame -> window -> FFT -> |X| -> dB) over
that block.  Multi-GPU: the recording is time-sharded, every rank owns a contiguous block plus an
(nfft - hop) halo it reads itself; no collective on the data path ("scaling": "weak").

  value      device-resident throughput (inputs already in HBM), CUDA-event timed, max over ranks
  e2e        same metric through the public host API (Engine.spectrogram on pinned HOST buffers):
             H2D of the step's samples and D2H of its dB image inside the timed region
  roofline   algorithmic bytes / kernel time against the measured HBM copy bandwidth
  cpu_baseline  the oracle (C FP64 port of the reference's Java path) on this box's host cores
  configs    the other BASELINE.json configurations (C2, C3, C4 one-GPU slice, C5), device-resident, each with
             its own roofline record (N = 1); at N > 1: config 4 time-sharded, one 2^30-sample cu8 block per rank
  sharded_matches_single / gather   (N > 1) the frames either side of every shard boundary computed in ONE unsharded
             call over the contiguous recording equal the rows the two neighbouring ranks produced, bit for bit;
             display assembly over NCCL timed on the device (full-resolution rows and the decimated canvas)
  e2e_mmap / e2e_file / e2e_canvas   the same step with the capture in a file-backed mmap (pageable in and out, the
             buffer the reference's SigMfHelper hands over), read from the file by the engine itself
             (sa_spectrogram_file), and as a display canvas (only W x H x 4 bytes come back)

--impl reference times that CPU port alone (the reference itself is Java; no JVM in the image).
--dump-outputs DIR writes a fixed, seeded sample of rows of the dB image of the last timed step (rank 0) as .npy files;
the recording is generated from fixed seeds, so two builds run with the same arguments can be compared row for row.
"""
import argparse
import json
import os
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NFFT, HOP, WINDOW, DATATYPE = 1024, 512, "hann", "cf32_le"
LOG2_SAMPLES_PER_GPU = 28
METRIC = "spectrogram Msamples/s (cf32, 1024-pt FFT)"
UNIT = "Msamples/s"
WORKLOAD = "cf32_le 2^%d samples/GPU, nfft 1024, Hann, hop 512 (50%% overlap), f32 dB out" % LOG2_SAMPLES_PER_GPU


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            # warm the two queries of the sampling loop (the first call of each is tens of ms)
            pynvml.nvmlDeviceGetClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.001)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def bind_near_gpu(torch, index):
    """Run this process on the CPUs of the GPU's NUMA node (sysfs local_cpulist) when the cpuset allows it, so that
    the pinned host buffers of the end-to-end leg are allocated on the memory next to the GPU's PCIe root (on a
    two-socket host the far node costs a third of the H2D/D2H rate).  Returns (previous affinity, info)."""
    try:
        p = torch.cuda.get_device_properties(index)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        base = "/sys/bus/pci/devices/" + bdf
        with open(base + "/local_cpulist") as f:
            txt = f.read().strip()
        try:
            with open(base + "/numa_node") as f:
                node = int(f.read())
        except Exception:
            node = None
        local = set()
        for part in txt.split(","):
            if part:
                lo, _, hi = part.partition("-")
                local.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        both = allowed & local
        info = {"gpu_numa_node": node, "allowed_cpus": len(allowed), "gpu_local_allowed_cpus": len(both), "bound": False}
        if both and both != allowed:
            os.sched_setaffinity(0, both)
            info["bound"] = True
        return allowed, info
    except Exception as e:                                    # no sysfs entry in this container: leave the affinity alone
        return None, {"error": str(e)[:100]}


REC_CHUNK = 1 << 24


def make_device_recording(torch, first, n, device, chunk=REC_CHUNK):
    """Samples [first, first + n) of THE synthetic recording (three tones of synth.TONES + white noise), generated on
    the device.  The recording is defined chunk by chunk (noise seeded by the chunk's index, tone phase from the
    absolute sample index), so every rank -- and the unsharded cross-check -- sees the same samples at the same
    positions.  `first` must be a multiple of the chunk."""
    from spectral_analyzer_b200 import synth
    assert first % chunk == 0
    out = torch.empty(2 * n, dtype=torch.float32, device=device)
    g = torch.Generator(device=device)
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        g.manual_seed(1000 + (first + s) // chunk)
        t = torch.arange(first + s, first + s + chunk, dtype=torch.float64, device=device)
        # always draw the whole chunk, then cut: a shorter draw would not be a prefix of the longer one
        re = torch.randn(chunk, generator=g, device=device, dtype=torch.float32) * synth.NOISE_SIGMA
        im = torch.randn(chunk, generator=g, device=device, dtype=torch.float32) * synth.NOISE_SIGMA
        for f, a in synth.TONES:
            ph = torch.remainder(f * t, 1.0) * (2 * 3.141592653589793)
            re += (a * torch.cos(ph)).float()
            im += (a * torch.sin(ph)).float()
        out[2 * s:2 * (s + m):2] = re[:m]
        out[2 * s + 1:2 * (s + m):2] = im[:m]
    return out


def cpu_port_throughput(n_samples, nthreads=0, min_seconds=0.0):
    """Times the oracle's spectrogram (C FP64 restatement of SpectralService.computeMagnitudes +
    the updateDisplay frame loop) on host cores; returns (Msamples/s, threads, seconds)."""
    import numpy as np
    from oracle import c_oracle as co
    from spectral_analyzer_b200 import synth
    block = synth.recording(1 << 20, DATATYPE, seed=1)
    raw = np.tile(block, max(1, n_samples >> 20))[: n_samples * 8]
    frames = (n_samples - NFFT) // HOP + 1
    threads = nthreads if nthreads > 0 else (len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count())
    co.spectrogram(raw[: 8 * (1 << 16)], DATATYPE, 0, NFFT, HOP, WINDOW, 64, nthreads=threads)     # warm
    reps, dt = 0, 0.0
    while reps < 1 or (dt < min_seconds and reps < 64):
        t0 = time.perf_counter()
        co.spectrogram(raw, DATATYPE, 0, NFFT, HOP, WINDOW, frames, nthreads=threads)
        dt += time.perf_counter() - t0
        reps += 1
    return reps * frames * HOP / dt / 1e6, threads, dt


def run_reference(args, rank):
    """Reference arm: the CPU implementation of the path (oracle port; the Java reference cannot
    run here) on the box's host cores, all threads."""
    if rank != 0:
        return
    n = 1 << 25          # bounded sample per step: 2^25 samples = 65535 frames (the size at which the port peaks)
    vals = []
    threads = 0
    for i in range(args.warmup + args.steps):
        v, threads, dt = cpu_port_throughput(n)
        if i >= args.warmup:
            vals.append((v, dt))
        if sum(d for _, d in vals) > 150:
            break
    ms = 1e3 * sum(d for _, d in vals) / len(vals)
    value = sum(v for v, _ in vals) / len(vals)
    sample = "2^25 samples per step (same cf32/1024/Hann/hop-512 parameters), %d steps" % len(vals)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(vals), "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def timed_ms(torch, fn, steps, warmup=3):
    """Median CUDA-event time of `fn` (launched on torch's current stream) over `steps` runs."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    t = sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(steps))
    return t[len(t) // 2]


DUMP_ROWS = 8192        # 8192 rows x 1024 bins x 4 B = 32 MiB


def dump_outputs(out_dir, d_out):
    """Writes what the timed step returns to its caller -- the [frames, NFFT] float32 dB image -- as a fixed sample: the
    first and last rows plus rows drawn with a fixed seed, so that two builds can be compared row for row."""
    import numpy as np
    import torch
    frames = d_out.shape[0]
    rows = np.arange(frames)
    if frames > DUMP_ROWS:
        inner = np.random.default_rng(0).choice(rows[1:-1], size=DUMP_ROWS - 2, replace=False)
        rows = np.sort(np.concatenate([[0], inner, [frames - 1]]))
    os.makedirs(out_dir, exist_ok=True)
    img = d_out.index_select(0, torch.from_numpy(rows).to(d_out.device)).cpu().numpy()
    np.save(os.path.join(out_dir, "spectrogram_db_rows.npy"), img)
    np.save(os.path.join(out_dir, "spectrogram_row_index.npy"), rows.astype(np.float64))


def other_configs(eng, steps, scale):
    """BASELINE.json configs[1..4] device-resident on one GPU, each with its own roofline record (algorithmic
    bytes of SURVEY.md 8d / median CUDA-event time / measured HBM peak).  Inputs + outputs of every case are far
    larger than L2."""
    import bench_configs as bc
    sc = lambda n: max(1 << 20, int(n * scale))
    cases = [
        lambda: bc.spectrogram_case(eng, "C2 ci16 4096 Blackman-Harris hop 4096, 2^30 samples", "ci16_le", sc(1 << 30), 4096, 4096,
                                    "blackman_harris", "f32", steps),
        lambda: bc.annotation_case(eng, sc(1 << 29), 500, min(1 << 20, sc(1 << 29) // 2), 16, steps),
        lambda: bc.annotation_case(eng, sc(1 << 29), 500, min(1 << 20, sc(1 << 29) // 2), 16, steps, want_iq=False),
        lambda: bc.spectrogram_case(eng, "C4 cu8 2048 rect -> RGBA heatmap, 2^31-sample slice", "cu8", sc(1 << 31), 2048, 2048,
                                    "rect", "rgba8", steps, colormap="Heatmap", sample_rate=2.4e6),
        lambda: bc.spectrogram_case(eng, "C5 cf64 65536 Hann FP64, 2^26 samples", "cf64_le", sc(1 << 26), 65536, 65536, "hann",
                                    "f64", steps),
        lambda: bc.spectrogram_case(eng, "C5b 16-bit WAV (ci16_le, 44-byte header) 1024 rect hop 1024, 2^28 samples (1 GiB in, 1 GiB out)", "ci16_le",
                                    sc(1 << 28), 1024, 1024, "rect", "f32", steps, byte_offset=44),
        lambda: bc.canvas_case(eng, sc(1 << 28), 1024, 512, 2048, 1024, "max", steps, host=False),
    ]
    out = []
    for fn in cases:
        try:
            r = fn()
        except Exception as ex:                         # a configuration that fails is reported, not hidden
            out.append({"error": str(ex)[:200]})
            continue
        rec = {"workload": r["config"], "ms": r["ms"], "Msamples_per_s": r["Msamples_per_s"], "kernel": r.get("kernel"),
               "roofline": {"bound": "hbm", "achieved": r["GBps"], "unit": "GB/s", "frac": r["roofline_frac"],
                            "alg_bytes": r["alg_bytes"], "peak_kind": r["peak_kind"]}}
        if "fft_flop_pipe_frac" in r:          # nominal FFT flops against the FP32 / FP64 FMA pipe peak (context for the HBM figure)
            rec["fft_flop_pipe_frac"] = r["fft_flop_pipe_frac"]
        out.append(rec)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2-samples", type=int, default=LOG2_SAMPLES_PER_GPU)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer legs")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configurations")
    ap.add_argument("--configs-scale", type=float, default=1.0, help="shrinks the sample counts of the other configurations")
    ap.add_argument("--sustained-steps", type=int, default=400,
                    help="extra back-to-back steps timed as one region to show the power-capped rate (0: skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed sample of rank 0's dB image from the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import ctypes as C
    import numpy as np
    import torch
    import torch.distributed as dist
    import spectral_analyzer_b200 as sa
    from spectral_analyzer_b200 import _capi, sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([float(x)], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n = 1 << args.log2_samples
    chunk = min(REC_CHUNK, n)
    halo = NFFT - HOP
    # rank r owns samples [r*n, (r+1)*n) of the recording and reads the halo that follows it
    n_local = n + (halo if rank < world - 1 else 0)
    frames = (n_local - NFFT) // HOP + 1
    d_iq = make_device_recording(torch, rank * n, n_local, device, chunk)
    d_out = torch.empty((frames, NFFT), dtype=torch.float32, device=device)
    eng = sa.Engine(local_rank)
    params = eng.make_params(DATATYPE, NFFT, HOP, WINDOW, n_frames=frames)
    stream = torch.cuda.current_stream().cuda_stream
    iq_bytes, out_bytes = d_iq.numel() * 4, d_out.numel() * 4

    def step():
        eng.spectrogram_device(d_iq.data_ptr(), iq_bytes, params, d_out.data_ptr(), out_bytes, stream)

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    launches0 = eng.kernel_launches
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    sampler.start()
    ev[0].record()
    for i in range(args.steps):
        step()
        ev[i + 1].record()
    barrier()
    sampler.stop_flag = True
    sampler.join()
    launches = eng.kernel_launches - launches0
    kernel_name = eng.last_kernel              # what the engine actually launched (sa_last_kernel_name), not a literal
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_out)
    per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    ms = max_over_ranks(ev[0].elapsed_time(ev[args.steps]) / args.steps)
    samples_per_step_local = frames * HOP
    tot = torch.tensor([float(samples_per_step_local)], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    value = tot.item() / (ms * 1e-3) / 1e6

    # roofline of the (single) kernel of the step: algorithmic bytes = every input byte once +
    # every output byte once (SURVEY 8d: 8 + 4*nfft/hop = 16 B per input sample)
    alg_bytes = n_local * 8 + frames * NFFT * 4
    kern_ms = sum(per_step) / len(per_step)            # average launch duration (one launch per step)
    kern_best, kern_median = min(per_step), sorted(per_step)[len(per_step) // 2]
    peak, peak_kind = hbm_peak()
    achieved = alg_bytes / (kern_ms * 1e-3) / 1e9
    # DRAM bytes of one launch: NOT measured in this run (that needs the profiler); the figure of the committed
    # ncu capture of the same kernel is carried with its source, and only when the kernel name still matches
    traffic, traffic_source = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        if tj.get("kernel") == kernel_name and n == 1 << LOG2_SAMPLES_PER_GPU:
            traffic = tj.get("spectrogram_f32_1024_cf32_hann_bytes_per_launch")
            traffic_source = tj.get("source")
    except Exception:
        pass

    # ---- N > 1: does the sharded image equal the unsharded one?  Rank r (< N-1) takes the contiguous span of the
    # recording around its right boundary (its last chunk + the next rank's first chunk, regenerated from the
    # recording's definition), computes the 64 frames before and the 64 frames after the boundary in ONE call, and
    # compares them bit for bit with its own last 64 rows and the next rank's first 64 rows.
    sharded = None
    if world > 1:
        kb = min(64, frames // 2)
        first_rows = [torch.empty((kb, NFFT), dtype=torch.float32, device=device) for _ in range(world)]
        dist.all_gather(first_rows, d_out[:kb].contiguous())
        ok = 1
        if rank < world - 1:
            span = make_device_recording(torch, (rank + 1) * n - chunk, 2 * chunk, device, chunk)
            ref = torch.empty((2 * kb, NFFT), dtype=torch.float32, device=device)
            # frames rank r owns end at frame n/HOP - 1 of its block: sample (rank+1)*n - HOP; kb of them, then kb of the next
            q = eng.make_params(DATATYPE, NFFT, HOP, WINDOW, n_frames=2 * kb, start_sample=chunk - kb * HOP)
            eng.spectrogram_device(span.data_ptr(), span.numel() * 4, q, ref.data_ptr(), ref.numel() * 4, stream)
            torch.cuda.synchronize()
            ok = int(torch.equal(ref[:kb], d_out[frames - kb:]) and torch.equal(ref[kb:], first_rows[rank + 1]))
            del span, ref
        t_ok = torch.tensor([ok], device=device, dtype=torch.int32)
        dist.all_reduce(t_ok, op=dist.ReduceOp.MIN)
        sharded = {"sharded_matches_single": bool(t_ok.item()),
                   "check": "%d boundaries x (%d + %d) frames across the boundary, one unsharded call over the contiguous span "
                            "vs the two ranks' rows, bit-exact" % (world - 1, kb, kb)}
        del first_rows

    # ---- N > 1: display assembly over NCCL, device-timed (outside the headline's timed region; SURVEY 8e)
    gather = None
    if world > 1:
        total_frames = int(tot.item()) // HOP
        def run_rows():
            return sharding.gather_rows(d_out, total_frames, dst=0)
        full = run_rows()                                   # warm-up: NCCL channels, allocator
        del full
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        full = run_rows()
        e1.record()
        barrier()
        rows_ms = max_over_ranks(e0.elapsed_time(e1))
        rows_bytes = (world - 1) * frames * NFFT * 4
        del full
        torch.cuda.empty_cache()
        W, H = 2048, 1024
        c0, c1, _, _ = sharding.canvas_columns(W, 1, world, rank)
        cols = c1 - c0
        fpc = frames // max(cols, 1)
        tile = torch.empty((H, cols), device=device, dtype=torch.int32)
        pc = eng.make_params(DATATYPE, NFFT, HOP, WINDOW, colormap="Heatmap", sample_rate=2.4e6)
        L = _capi.lib()
        def render():
            _capi.check(L.sa_render_canvas_device(eng.handle, d_iq.data_ptr(), iq_bytes, C.byref(pc), cols, H, fpc,
                                                  _capi.REDUCE["max"], tile.data_ptr(), stream))
        tile4 = tile.view(torch.uint8).view(H, cols, 4)
        render()
        sharding.gather_canvas(tile4, W, dst=0)
        barrier()
        e2 = torch.cuda.Event(enable_timing=True)
        e0.record()
        render()
        e1.record()
        canvas = sharding.gather_canvas(tile4, W, dst=0)
        e2.record()
        barrier()
        gather = {"rows_ms": round(rows_ms, 3), "rows_bytes": int(rows_bytes),
                  "rows_GBps_into_rank0": round(rows_bytes / rows_ms / 1e6, 1),
                  "canvas_render_ms": round(max_over_ranks(e0.elapsed_time(e1)), 3),
                  "canvas_ms": round(max_over_ranks(e1.elapsed_time(e2)), 3), "bytes": W * H * 4,
                  "canvas": "%dx%d max-pooled, every rank renders its columns (%d frames each) from its own block" % (W, H, fpc),
                  "api": "sharding.gather_rows / gather_canvas (dist.gather over NCCL), CUDA-event timed, max over ranks"}
        del canvas, tile

    # ---- end-to-end legs: public host API, H2D + D2H inside the timed region
    e2e = e2e_mmap = e2e_file = e2e_canvas = None
    if not args.no_e2e:
        prev_aff, numa = bind_near_gpu(torch, local_rank)
        h_iq = torch.empty(d_iq.numel(), dtype=torch.float32, pin_memory=True)
        h_iq.copy_(d_iq)
        h_out = torch.empty((frames, NFFT), dtype=torch.float32, pin_memory=True)
        h_iq_np, h_out_np = h_iq.numpy(), h_out.numpy()
        e2e_steps = max(3, min(args.steps, 8))

        def host_leg(fn, steps, warm=2):
            for _ in range(warm):
                fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            barrier()
            return max_over_ranks((time.perf_counter() - t0) / steps)

        dt = host_leg(lambda: eng.spectrogram(h_iq_np, DATATYPE, NFFT, frames, hop=HOP, window=WINDOW, out=h_out_np), e2e_steps)
        e2e = {"value": round(tot.item() / dt / 1e6, 3), "unit": UNIT,
               "h2d_bytes_per_step": int(n_local * 8), "d2h_bytes_per_step": int(frames * NFFT * 4),
               "ms_per_step": round(dt * 1e3, 3), "steps": e2e_steps,
               "api": "Engine.spectrogram (sa_spectrogram C-ABI), pinned host in/out"}
        e2e["matches_device_path"] = bool(torch.equal(h_out.to(device), d_out))
        e2e["numa"] = numa

        # display canvas of the same block: all samples go in, only W x H x 4 bytes come back
        W, H = 2048, 1024
        fpc = max(1, frames // W)
        dt = host_leg(lambda: eng.render_canvas(h_iq_np, DATATYPE, NFFT, W, H, 2.4e6, hop=HOP, window=WINDOW,
                                                frames_per_column=fpc, reduce="max", colormap="Heatmap"), 3, warm=1)
        e2e_canvas = {"value": round(world * W * fpc * HOP / dt / 1e6, 3), "unit": UNIT, "ms_per_step": round(dt * 1e3, 3),
                      "h2d_bytes_per_step": int(n_local * 8), "d2h_bytes_per_step": W * H * 4,
                      "api": "Engine.render_canvas (sa_render_canvas), %dx%d max-pooled, pinned host in" % (W, H)}

        # the app's own input: the .sigmf-data file.  (a) file-backed mmap in, pageable array out -- the
        # MappedByteBuffer of SigMfHelper.java:78-84, which cannot be page-locked; (b) the engine reads the file itself
        tmpdir = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
        # a unique name: another user's file of the same name in the shared directory must not break this leg
        fd, path = tempfile.mkstemp(prefix="sa_bench_rank%d_" % rank, suffix=".sigmf-data", dir=tmpdir)
        os.close(fd)
        try:
            st = os.statvfs(tmpdir)
            if st.f_bavail * st.f_frsize < 2 * world * n_local * 8:
                raise OSError("not enough space in %s" % tmpdir)
            h_iq_np.tofile(path)
            mm = np.memmap(path, dtype=np.uint8, mode="r")
            out_pageable = np.empty((frames, NFFT), np.float32)
            dt = host_leg(lambda: eng.spectrogram(mm, DATATYPE, NFFT, frames, hop=HOP, window=WINDOW, out=out_pageable), 3, warm=1)
            e2e_mmap = {"value": round(tot.item() / dt / 1e6, 3), "unit": UNIT, "ms_per_step": round(dt * 1e3, 3),
                        "h2d_bytes_per_step": int(n_local * 8), "d2h_bytes_per_step": int(frames * NFFT * 4),
                        "matches_device_path": bool(np.array_equal(out_pageable, h_out_np)),
                        "api": "Engine.spectrogram on np.memmap of the data file in %s (page cache warm), pageable "
                               "float32 array out: both directions staged through the engine's pinned ring" % tmpdir}
            del mm, out_pageable
            h_out_np[:] = 0
            dt = host_leg(lambda: eng.spectrogram_file(path, DATATYPE, NFFT, frames, hop=HOP, window=WINDOW, out=h_out_np), 3, warm=1)
            e2e_file = {"value": round(tot.item() / dt / 1e6, 3), "unit": UNIT, "ms_per_step": round(dt * 1e3, 3),
                        "h2d_bytes_per_step": int(n_local * 8), "d2h_bytes_per_step": int(frames * NFFT * 4),
                        "matches_device_path": bool(torch.equal(h_out.to(device), d_out)),
                        "api": "Engine.spectrogram_file (sa_spectrogram_file: parallel pread into the pinned ring), pinned out"}
        except Exception as ex:
            e2e_mmap = e2e_mmap or {"unavailable": str(ex)[:160]}
        finally:
            try:
                os.unlink(path)
            except OSError:
                pass
        if prev_aff is not None and numa.get("bound"):
            os.sched_setaffinity(0, prev_aff)
        del h_iq, h_out, h_iq_np, h_out_np

    # ---- sustained leg: the same step back to back for ~0.4 s; on a 1 kW part the SM clock drops under
    # sw_power_cap, so this is the rate a long recording sees (reported beside, not instead of, `value`)
    sustained = None
    if args.sustained_steps > 0:
        s2 = ClockSampler(local_rank)
        s2.start()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.sustained_steps):
            step()
        e1.record()
        barrier()
        s2.stop_flag = True
        s2.join()
        ts = max_over_ranks(e0.elapsed_time(e1) / args.sustained_steps)
        sustained = {"steps": args.sustained_steps, "ms_per_step": round(ts, 4),
                     "value": round(tot.item() / (ts * 1e-3) / 1e6, 3), "unit": UNIT,
                     "roofline_frac": round(alg_bytes / (ts * 1e-3) / 1e9 / peak, 4), "clocks": s2.summary()}

    # ---- the other BASELINE configurations
    configs = None
    del d_iq, d_out
    torch.cuda.empty_cache()
    if not args.no_configs:
        if world == 1:
            configs = other_configs(eng, 7, args.configs_scale)
        else:
            # config 4 as BASELINE.json states it: cu8 recording time-sharded over the ranks, 2^30 samples (2 GiB) each
            # -> 16 GiB at 8 GPUs; 2048-pt, hop 2048 (no halo), RGBA heatmap out; max over ranks
            n4 = max(1 << 20, int((1 << 30) * args.configs_scale))
            f4 = n4 // 2048
            g = torch.Generator(device=device)
            g.manual_seed(4000 + rank)
            raw = torch.randint(0, 256, (2 * n4,), device=device, dtype=torch.uint8, generator=g)
            out4 = torch.empty(f4 * 2048, device=device, dtype=torch.int32)
            p4 = eng.make_params("cu8", 2048, 2048, "rect", n_frames=f4, out="rgba8", colormap="Heatmap", sample_rate=2.4e6)
            barrier()
            ms4 = max_over_ranks(timed_ms(torch, lambda: eng.spectrogram_device(raw.data_ptr(), raw.numel(), p4, out4.data_ptr(),
                                                                                out4.numel() * 4, stream), 10))
            alg4 = 2 * n4 + f4 * 2048 * 4
            configs = [{"workload": "C4 cu8 2048 rect -> RGBA heatmap, time-sharded: 2^%d samples per GPU x %d GPUs (%.0f GiB recording)"
                                    % (n4.bit_length() - 1, world, world * 2 * n4 / 2 ** 30),
                        "ms": round(ms4, 4), "Msamples_per_s": round(world * f4 * 2048 / ms4 / 1e3, 1), "kernel": eng.last_kernel,
                        "roofline": {"bound": "hbm", "achieved": round(alg4 / ms4 / 1e6, 1), "unit": "GB/s (per GPU)",
                                     "frac": round(alg4 / ms4 / 1e6 / peak, 4), "alg_bytes": alg4, "peak_kind": peak_kind}}]
            del raw, out4

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        v1, _, dt1 = cpu_port_throughput(1 << 21, nthreads=1)
        # bounded sample: 2^25 samples repeated until about 4 s of wall time on all host threads
        log2n = 25
        vall, threads, dtall = cpu_port_throughput(1 << log2n, min_seconds=4.0)
        # second opinion (SURVEY 8d): numpy / pocketfft FP64 on one thread, same framing, window and dB form
        from spectral_analyzer_b200 import synth
        nn = 1 << 21
        xs = np.frombuffer(synth.recording(nn, DATATYPE, seed=1).tobytes(), np.complex64).astype(np.complex128)
        wnd = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(NFFT) / NFFT)
        t0 = time.perf_counter()
        fr = np.lib.stride_tricks.sliding_window_view(xs, NFFT)[::HOP] * wnd
        _ = np.fft.fftshift(20 * np.log10(np.abs(np.fft.fft(fr, axis=1)) + 1e-10), axes=1)
        v_np = fr.shape[0] * HOP / (time.perf_counter() - t0) / 1e6
        cpu = {"value": round(vall, 3), "unit": UNIT, "cores": threads, "kind": "port",
               "numpy_pocketfft_1thread_value": round(v_np, 3),
               "sample": "2^%d samples (repeated), same parameters, %.1f s on %d threads; 1 thread (the reference's FX-thread "
                         "concurrency): %.3f Msamples/s on 2^21 samples" % (log2n, dtall, threads, v1),
               "single_thread_value": round(v1, 3)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "datatype": DATATYPE, "nfft": NFFT, "hop": HOP, "window": WINDOW,
                       "samples_per_gpu": n, "frames_per_gpu": frames, "sharding": "time blocks + %d-sample halo" % halo,
                       "l2": "inputs (2 GiB) and outputs (2 GiB) per step are far larger than the 126 MB L2",
                       "reference_sample": "the --impl reference arm runs the same parameters on 2^25 samples per step "
                                           "(bounded CPU time); the metric is per sample"},
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_source,
                         "peak_kind": peak_kind,
                         "alg_bytes_per_launch": int(alg_bytes), "kernel_ms": round(kern_ms, 4),
                         "kernel_ms_best": round(kern_best, 4), "kernel_ms_median": round(kern_median, 4),
                         "kernel": kernel_name},
            "clocks": sampler.summary(),
            "gpu_launches": int(launches),
        }
        # the FP32 pipe bound beside the HBM one (SURVEY 8d): 5 nfft log2(nfft) / hop + 6 flop per input sample against
        # 148 SMs x 128 FMA lanes x 2 flop at the SM clock sampled during the run
        import math
        flops_per_sample = 5.0 * NFFT * math.log2(NFFT) / HOP + 6.0
        sm_mhz = (line["clocks"] or {}).get("sm_mhz") or 1965
        fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
        fp32_ach = samples_per_step_local * flops_per_sample / (kern_ms * 1e-3) / 1e12
        line["fp32_pipe"] = {"flops_per_sample": round(flops_per_sample, 1), "achieved": round(fp32_ach, 2),
                             "peak": round(fp32_peak, 1), "unit": "TFLOP/s", "frac": round(fp32_ach / fp32_peak, 4)}
        for k, v in (("e2e", e2e), ("e2e_mmap", e2e_mmap), ("e2e_file", e2e_file), ("e2e_canvas", e2e_canvas),
                     ("sustained", sustained), ("configs", configs), ("cpu_baseline", cpu)):
            if v:
                line[k] = v
        if sharded:
            line.update(sharded)
        if gather:
            line["gather"] = gather
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    eng.close()


if __name__ == "__main__":
    main()
