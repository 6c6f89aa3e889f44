"""Spectrum-trace timings on the GPU (device-resident input larger than L2, CUDA events, the variants of one workload
alternated within one call), next to the spectrogram rows and the max-pooled canvas of the same frames.

    python tools/trace_bench.py [--reps 20] [--out profiles/trace_bench.json]

Prints one JSON line per measurement and writes them all, with the card name and power limit, to --out."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import spectral_analyzer_b200 as sa  # noqa: E402
from spectral_analyzer_b200 import _capi  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def alternate(fns, reps):
    """fns: {name: callable enqueuing work on the current stream}; round-robin, median ms per name"""
    for f in fns.values():
        f()
    torch.cuda.synchronize()
    times = {k: [] for k in fns}
    for _ in range(reps):
        for k, f in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            f()
            b.record()
            b.synchronize()
            times[k].append(a.elapsed_time(b))
    return {k: float(np.median(v)) for k, v in times.items()}


def trace_fn(eng, d_iq, nbytes, p, F, stats, stream):
    n_rows = -(-p.n_frames // F)
    esz = 8 if p.out_kind == _capi.OUT_F64_DB else 4
    outs = {s: torch.empty(n_rows * p.nfft * esz, dtype=torch.uint8, device="cuda") for s in stats}
    ptr = [outs[s].data_ptr() if s in outs else None for s in ("mean", "max", "min")]
    return lambda: eng.spectrum_trace_device(d_iq.data_ptr(), nbytes, p, F, *ptr, n_rows * p.nfft * esz, stream)


def rows_fn(eng, d_iq, nbytes, p, stream):
    esz = 8 if p.out_kind == _capi.OUT_F64_DB else 4
    out = torch.empty(p.n_frames * p.nfft * esz, dtype=torch.uint8, device="cuda")
    return lambda: eng.spectrogram_device(d_iq.data_ptr(), nbytes, p, out.data_ptr(), out.numel(), stream)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "trace_bench.json"))
    a = ap.parse_args()
    eng = sa.Engine(0)
    stream = torch.cuda.current_stream().cuda_stream
    res = {"card": card(), "results": []}

    def emit(rec):
        print(json.dumps(rec), flush=True)
        res["results"].append(rec)

    # headline: 2^28 cf32 samples (2 GiB, far beyond the 126 MB L2), 1024-point Hann, hop 512
    n, nfft, hop = 1 << 28, 1024, 512
    frames = (n - nfft) // hop + 1
    d_iq = torch.randn(2 * n, device="cuda", dtype=torch.float32).mul_(0.1)
    p = eng.make_params("cf32_le", nfft, hop, "hann", n_frames=frames)
    W, H = 2048, 1024
    fpc = frames // W
    pc = eng.make_params("cf32_le", nfft, hop, "hann", colormap="Heatmap", sample_rate=2.4e6)
    canvas = torch.empty(W * H * 4, dtype=torch.uint8, device="cuda")
    fns = {"trace mean, 1 row": trace_fn(eng, d_iq, n * 8, p, frames, ("mean",), stream),
           "trace max, 1 row": trace_fn(eng, d_iq, n * 8, p, frames, ("max",), stream),
           "trace mean+max+min, 1 row": trace_fn(eng, d_iq, n * 8, p, frames, ("mean", "max", "min"), stream),
           "trace mean+max+min, 2048 rows": trace_fn(eng, d_iq, n * 8, p, -(-frames // 2048), ("mean", "max", "min"), stream),
           "spectrogram rows f32": rows_fn(eng, d_iq, n * 8, p, stream),
           "canvas max 2048 columns": lambda: _capi.check(_capi.lib().sa_render_canvas_device(
               eng.handle, d_iq.data_ptr(), n * 8, C.byref(pc), W, H, fpc, _capi.REDUCE["max"], canvas.data_ptr(), stream))}
    fns["trace max, 1 row"]()
    torch.cuda.synchronize()
    kernel = eng.last_kernel
    for k, ms in alternate(fns, a.reps).items():
        emit({"workload": "cf32 2^28 1024 Hann hop 512 (%d frames)" % frames, "variant": k, "ms": round(ms, 4),
              "Msamples_per_s": round(frames * hop / ms / 1e3, 1), "trace_kernel": kernel})
    del d_iq, fns
    torch.cuda.empty_cache()

    # C4 shape: cu8 2048 rect; C5: cf64 65536 Hann on the FP64 path
    for name, dt, n, nfft, win, prec, raw in (
            ("C4 cu8 2048 rect", "cu8", 1 << 30, 2048, "rect", "auto",
             lambda n: torch.randint(0, 255, (2 * n,), device="cuda", dtype=torch.uint8)),
            ("C5 cf64 65536 Hann FP64", "cf64_le", 1 << 26, 65536, "hann", "f64",
             lambda n: torch.randn(2 * n, device="cuda", dtype=torch.float64).mul_(0.1))):
        d_iq = raw(n)
        nb = d_iq.numel() * d_iq.element_size()
        frames = (n - nfft) // nfft + 1
        out = "f64" if prec == "f64" else "f32"
        p = eng.make_params(dt, nfft, nfft, win, n_frames=frames, out=out, precision=prec)
        fns = {"trace mean, 1 row": trace_fn(eng, d_iq, nb, p, frames, ("mean",), stream),
               "trace mean+max+min, 1 row": trace_fn(eng, d_iq, nb, p, frames, ("mean", "max", "min"), stream),
               "spectrogram rows %s" % out: rows_fn(eng, d_iq, nb, p, stream)}
        fns["trace mean, 1 row"]()
        torch.cuda.synchronize()
        kernel = eng.last_kernel
        for k, ms in alternate(fns, a.reps).items():
            emit({"workload": name, "variant": k, "ms": round(ms, 4), "Msamples_per_s": round(frames * nfft / ms / 1e3, 1),
                  "trace_kernel": kernel})
        del d_iq, fns
        torch.cuda.empty_cache()

    # host entry: 2^28 cf32 samples in pinned and in pageable memory, three statistics, one row
    n, nfft, hop = 1 << 28, 1024, 512
    frames = (n - nfft) // hop + 1
    pinned = torch.randn(2 * n, dtype=torch.float32).mul_(0.1).pin_memory()
    pageable = pinned.numpy().copy()
    for tag, buf in (("pinned", pinned.numpy()), ("pageable", pageable)):
        eng.spectrum_trace(buf, "cf32_le", nfft, frames, hop=hop, window="hann", stats=("mean", "max", "min"))
        ts = []
        for _ in range(max(3, a.reps // 4)):
            t0 = time.perf_counter()
            eng.spectrum_trace(buf, "cf32_le", nfft, frames, hop=hop, window="hann", stats=("mean", "max", "min"))
            ts.append((time.perf_counter() - t0) * 1e3)
        emit({"workload": "host entry cf32 2^28 1024 Hann hop 512", "variant": tag + ", mean+max+min, 1 row",
              "ms": round(float(np.median(ts)), 2), "Msamples_per_s": round(n / np.median(ts) / 1e3, 1)})
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
