"""Persistence-spectrum timings on the GPU (device-resident input larger than L2, CUDA events, the variants of one
workload alternated within one call): persistence against the F32 rows path, a one-row MAX trace and the unfused
baseline it replaces (F32 rows, then torch.bucketize + torch.bincount over level * nfft + bin on the GPU).

    python tools/persistence_bench.py [--reps 15] [--out profiles/persistence_bench.json] [--headline-only]

Prints one JSON line per measurement and writes them all, with the card name, power limit and max SM clock, to --out.
SA_ENGINE_LIB selects another build of the library (the chunk-size ablation of DESIGN.md N5)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import spectral_analyzer_b200 as sa  # noqa: E402
from trace_bench import alternate, rows_fn, trace_fn  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def persistence_fn(eng, d_iq, nbytes, p, n_levels, lo, hi, stream):
    counts = torch.empty(n_levels * p.nfft, dtype=torch.int32, device="cuda")
    return lambda: eng.spectrum_persistence_device(d_iq.data_ptr(), nbytes, p, n_levels, lo, hi, counts.data_ptr(),
                                                   counts.numel() * 4, stream)


def unfused_fn(eng, d_iq, nbytes, p, n_levels, lo, hi, stream):
    """A timing baseline for the route persistence replaces, not a bit-equivalent histogram: F32 rows, then in torch
    bucketize against FP32 level boundaries lo + j (hi - lo) / n (not the engine's quantizer) and a count of
    level * nfft + bin (torch.histc with one bin per index, exact below 2^24 bins; torch.bincount, which sizes its output
    from the data, failed on the C4 shape with "Storage size calculation overflowed")."""
    rows = torch.empty(p.n_frames, p.nfft, dtype=torch.float32, device="cuda")
    bounds = torch.tensor([lo + j * (hi - lo) / n_levels for j in range(1, n_levels)], dtype=torch.float32, device="cuda")
    k = torch.arange(p.nfft, device="cuda")

    step = max(1, (1 << 27) // p.nfft)             # frames per torch pass (bounds the int64 temporaries)

    def run():
        eng.spectrogram_device(d_iq.data_ptr(), nbytes, p, rows.data_ptr(), rows.numel() * 4, stream)
        counts = torch.zeros(n_levels * p.nfft, dtype=torch.int64, device="cuda")
        for f0 in range(0, p.n_frames, step):
            lv = torch.bucketize(rows[f0:f0 + step], bounds, right=True)
            idx = (lv * p.nfft + k).view(-1).float()
            counts += torch.histc(idx, bins=n_levels * p.nfft, min=0, max=n_levels * p.nfft).long()
        return counts
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "persistence_bench.json"))
    ap.add_argument("--headline-only", action="store_true")
    a = ap.parse_args()
    eng = sa.Engine(0)
    stream = torch.cuda.current_stream().cuda_stream
    res = {"card": card(), "library": os.path.basename(os.environ.get("SA_ENGINE_LIB", "libsa_engine.so")), "results": []}

    def emit(rec):
        print(json.dumps(rec), flush=True)
        res["results"].append(rec)

    # headline shape: 2^28 cf32 samples (2 GiB, far beyond the 126 MB L2), 1024-point Hann, hop 512, 256 levels;
    # C4: 2^30 cu8, 2048 rect; C5: 2^26 cf64, 65536 Hann on the FP64 path
    shapes = [("cf32 2^28 1024 Hann hop 512, 256 levels", "cf32_le", 1 << 28, 1024, 512, "hann", "auto", 256, -60.0, 20.0,
               lambda n: torch.randn(2 * n, device="cuda", dtype=torch.float32).mul_(0.1)),
              ("C4 cu8 2^30 2048 rect, 256 levels", "cu8", 1 << 30, 2048, 2048, "rect", "auto", 256, -20.0, 80.0,
               lambda n: torch.randint(0, 255, (2 * n,), device="cuda", dtype=torch.uint8)),
              ("C5 cf64 2^26 65536 Hann FP64, 256 levels", "cf64_le", 1 << 26, 65536, 65536, "hann", "f64", 256, -40.0,
               40.0, lambda n: torch.randn(2 * n, device="cuda", dtype=torch.float64).mul_(0.1))]
    for name, dt, n, nfft, hop, win, prec, n_levels, lo, hi, raw in shapes[:1] if a.headline_only else shapes:
        d_iq = raw(n)
        nb = d_iq.numel() * d_iq.element_size()
        frames = (n - nfft) // hop + 1
        p = eng.make_params(dt, nfft, hop, win, n_frames=frames, precision=prec)
        pr = eng.make_params(dt, nfft, hop, win, n_frames=frames, precision=prec)      # rows: F32 dB
        fns = {"persistence": persistence_fn(eng, d_iq, nb, p, n_levels, lo, hi, stream),
               "spectrogram rows f32": rows_fn(eng, d_iq, nb, pr, stream),
               "trace max, 1 row": trace_fn(eng, d_iq, nb, pr, frames, ("max",), stream)}
        if name.startswith("cf32"):                 # where the time goes: the histogram's shared memory per CTA
            for nl in (2, 37):
                fns["persistence, %d levels" % nl] = persistence_fn(eng, d_iq, nb, p, nl, lo, hi, stream)
        if not a.headline_only:
            fns["unfused timing baseline: rows f32 + torch bucketize/histc"] = unfused_fn(eng, d_iq, nb, pr, n_levels, lo, hi, stream)
        fns["persistence"]()
        torch.cuda.synchronize()
        kernel = eng.last_kernel
        for k, ms in alternate(fns, a.reps).items():
            emit({"workload": name, "frames": frames, "variant": k, "ms": round(ms, 4),
                  "Msamples_per_s": round(frames * hop / ms / 1e3, 1), "persistence_kernels": kernel})
        del d_iq, fns
        torch.cuda.empty_cache()

    if not a.headline_only:
        # host entry: 2^28 cf32 samples in pinned and in pageable memory, 256 levels
        n, nfft, hop = 1 << 28, 1024, 512
        frames = (n - nfft) // hop + 1
        pinned = torch.randn(2 * n, dtype=torch.float32).mul_(0.1).pin_memory()
        pageable = pinned.numpy().copy()
        for tag, buf in (("pinned", pinned.numpy()), ("pageable", pageable)):
            eng.spectrum_persistence(buf, "cf32_le", nfft, frames, 256, -60.0, 20.0, hop=hop, window="hann")
            ts = []
            for _ in range(max(3, a.reps // 3)):
                t0 = time.perf_counter()
                eng.spectrum_persistence(buf, "cf32_le", nfft, frames, 256, -60.0, 20.0, hop=hop, window="hann")
                ts.append((time.perf_counter() - t0) * 1e3)
            emit({"workload": "host entry cf32 2^28 1024 Hann hop 512, 256 levels", "variant": tag,
                  "ms": round(float(np.median(ts)), 2), "Msamples_per_s": round(n / np.median(ts) / 1e3, 1)})
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
