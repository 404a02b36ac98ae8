"""Throughput of mridc_b200.espirit_maps (ESPIRiT coil maps) in slices/s, with the time of each stage.

Geometries: 15 x 320 x 320 and 16 x 640 x 320 (the fastMRI knee / brain shapes of bench.py) and 32 x 232 x 288, fully
sampled synthetic k-space (synth.make_batch), default parameters (cw 24, kw 6, threshold 0.02, crop 0.95, 100 iterations).
The end-to-end time is taken with CUDA events around espirit_maps; the stages (Gram kernel, eigh, taps, inverse FFT,
power iterations) with events around the same calls made one by one.  Prints one JSON line per geometry, with the card
name and its power limit read in the same run.

    python tools/bench_espirit.py [--reps 3] [--out results/bench_espirit.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

GEOMS = [(8, 15, 320, 320), (4, 16, 640, 320), (4, 32, 232, 288)]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        return out.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "%s (nvidia-smi unavailable: %s)" % (torch.cuda.get_device_name(), e)


def stages(y, cw=24, kw=6, threshold=0.02, crop=0.95, max_iter=100):
    """espirit_maps split into its calls, one CUDA event between each -> dict stage -> ms."""
    from mridc_b200 import _lib, espirit

    lib, base = espirit.load(), _lib.load()
    B, C, H, W, _ = y.shape
    N, P = C * kw * kw, C * (C + 1) // 2
    st = _lib.stream_ptr()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
    ev[0].record()
    gram = torch.empty(B, N, N, 2, dtype=torch.float64, device="cuda")
    espirit.check(lib.mrbe_calib_gram(_lib.ptr(y), _lib.ptr(gram), B, C, H, W, cw, kw, 1, st))
    ev[1].record()
    g = torch.view_as_complex(gram)
    vecs = torch.empty(B, N, N, dtype=torch.complex128, device="cuda")
    rank = torch.empty(B, dtype=torch.int32, device="cuda")
    for b in range(B):
        e, V = torch.linalg.eigh(g[b])
        s = e.clamp_min(0).sqrt()
        rank[b] = (s > threshold * s[-1]).sum()
        vecs[b] = V.mT
    ev[2].record()
    chunk = max(1, min(B, espirit.G_CHUNK_BYTES // (P * H * W * 8)))
    gbuf = torch.empty(chunk, P, H, W, 2, device="cuda")
    maps = torch.empty(B, C, H, W, 2, device="cuda")
    lam = torch.empty(B, H, W, device="cuda")
    t = {"taps": 0.0, "fft": 0.0, "power": 0.0}
    for b0 in range(0, B, chunk):
        n = min(chunk, B - b0)
        a = torch.cuda.Event(enable_timing=True)
        a.record()
        espirit.check(lib.mrbe_kernel_taps(_lib.ptr(vecs[b0]), _lib.ptr(rank[b0:]), _lib.ptr(gbuf), n, C, H, W, kw, 1, st))
        ev[3].record()
        _lib.check(base.mrb_fft2_c2c(_lib.ptr(gbuf), _lib.ptr(gbuf), n * P, H, W, 1, 1, 2, st))
        ev[4].record()
        espirit.check(lib.mrbe_power_maps(_lib.ptr(gbuf), _lib.ptr(maps[b0]), _lib.ptr(lam[b0]), n, C, H, W, max_iter,
                                          crop, st))
        ev[5].record()
        torch.cuda.synchronize()
        t["taps"] += a.elapsed_time(ev[3])
        t["fft"] += ev[3].elapsed_time(ev[4])
        t["power"] += ev[4].elapsed_time(ev[5])
    torch.cuda.synchronize()
    t["gram"] = ev[0].elapsed_time(ev[1])
    t["eigh"] = ev[1].elapsed_time(ev[2])
    return t, maps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_espirit.py measures on a CUDA device"
    import mridc_b200 as mb
    from mridc_b200 import synth

    info = card()
    rows = []
    for B, C, H, W in GEOMS:
        y = synth.make_batch(B, C, H, W, centered=True, normalization="ortho")["kspace"].cuda()
        ref = mb.espirit_maps(y)  # warm-up (module load, eigh workspaces, FFT plans)
        torch.cuda.synchronize()
        e2e = []
        for _ in range(args.reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            mb.espirit_maps(y)
            b.record()
            torch.cuda.synchronize()
            e2e.append(a.elapsed_time(b))
        st, maps = stages(y)
        assert torch.equal(maps, ref), "the staged run differs from espirit_maps"
        ms = sorted(e2e)[len(e2e) // 2]
        row = {"geometry": "%dx%dx%d" % (C, H, W), "batch": B, "ms_per_batch": round(ms, 3),
               "slices_per_s": round(1000.0 * B / ms, 2), "e2e_ms_all": [round(v, 3) for v in e2e],
               "stage_ms": {k: round(v, 3) for k, v in st.items()},
               "power_share": round(st["power"] / sum(st.values()), 4), "card": info}
        print(json.dumps(row), flush=True)
        rows.append(row)
        del y, ref, maps
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    main()
