"""Throughput of mridc_b200.pics.l1_wavelet_recon (PICS, l1-wavelet FISTA) in slices/s, and where an iteration goes.

Geometries: 15 x 320 x 320 at B = 8 and 16, 16 x 640 x 320 at B = 4 (the fastMRI knee / brain shapes of bench.py); synthetic
k-space (synth.make_batch) under a 4x equispaced column mask, 100 iterations, lamda = 0.01 max |Psi E^H y|.  Timing:
  - end to end: CUDA events around l1_wavelet_recon (median of --reps);
  - per iteration: the same loop run with CUDA events around each data-term gradient and each proximal step;
  - the proximal step's algorithmic bytes (computed from the shapes: every level reads and writes its band once, level 1
    also reads the gradient and x_k and writes z) over its time, as a fraction of the HBM bandwidth of a device-to-device
    copy measured in the same run;
  - a CPU baseline: one slice, the same iterations in fp32 torch on the CPU (torch.fft, Psi as dense 1-D matrices).
Prints one JSON line per geometry with the card name and power limit read in the same run.

    python tools/bench_pics.py [--reps 3] [--cpu-iters 100] [--out results/bench_pics.json]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

GEOMS = [(8, 15, 320, 320), (16, 15, 320, 320), (4, 16, 640, 320)]
ITERS = 100
LAMBDA_FRAC = 0.01


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        return out.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "%s (nvidia-smi unavailable: %s)" % (torch.cuda.get_device_name(), e)


def copy_bandwidth(nbytes=4 << 30, reps=10):
    """Device-to-device copy rate in bytes/s (read + write), median of reps; the HBM peak this run compares against."""
    a = torch.empty(nbytes // 2, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / 1e3)
    del a, b
    torch.cuda.empty_cache()
    return nbytes / sorted(ts)[len(ts) // 2]


def prox_bytes(B, H, W, levels):
    """Algorithmic bytes of one mrbp_fista_step: level 1 analysis reads z and grad channels 2-3 and writes the band
    (3 x 8 B per pixel), level 1 synthesis reads the band and x_k and writes x and z (4 x 8 B); every other level reads
    and writes its band once in each direction (4 x 8 B per band sample)."""
    n = B * H * W
    total = 24 * n + 32 * n
    for l in range(2, levels + 1):
        total += 32 * (n >> (2 * (l - 1)))
    return total


def lam_for(y, S, mask):
    from mridc_b200 import _ops, pics

    eh = _ops.sens_reduce(y, S, True, "ortho")  # E^H y = -grad f(0) for a 0/1 mask
    return LAMBDA_FRAC * float(pics.dwt(eh).pow(2).sum(-1).sqrt().amax())


def split(y, S, mask, lam):
    """The solver loop with CUDA events around each gradient and each proximal step -> (dc ms, prox ms) per iteration."""
    from mridc_b200 import _lib, _ops, pics

    B, C, H, W, _ = y.shape
    lib, levels = pics.load(), pics.wavelet_levels(H, W)
    m = _ops.canonical_mask(mask, B, H, W)[0]
    alpha = pics.step_size(S, m)
    yh = _ops.dc_hybrid_prepare(y, m, True)
    x = torch.zeros(B, H, W, 2, device="cuda")
    z = torch.zeros_like(x)
    g = torch.empty(B, 4, H, W, device="cuda")
    ws, n = pics._workspace(B, H, W, y.device)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * ITERS + 1)]
    t = 1.0
    ev[0].record()
    for k in range(ITERS):
        _ops.dc_rim_grad(z, y, S, m, 1.0, True, "ortho", out=g, y_hybrid=yh)
        ev[2 * k + 1].record()
        tn = (1 + math.sqrt(1 + 4 * t * t)) / 2
        pics.check(lib.mrbp_fista_step(_lib.ptr(z), _lib.ptr(g), _lib.ptr(alpha), lam, (t - 1) / tn, _lib.ptr(x), B, H,
                                       W, levels, _lib.ptr(ws), n, _lib.stream_ptr()))
        ev[2 * k + 2].record()
        t = tn
    torch.cuda.synchronize()
    dc = sum(ev[2 * k].elapsed_time(ev[2 * k + 1]) for k in range(ITERS)) / ITERS
    prox = sum(ev[2 * k + 1].elapsed_time(ev[2 * k + 2]) for k in range(ITERS)) / ITERS
    return dc, prox, x


def cpu_baseline(y, S, mask, lam, iters):
    """One slice, fp32 torch on the CPU, the same FISTA iterations -> seconds."""
    from mridc_b200 import pics

    y = torch.view_as_complex(y[:1].cpu().contiguous())
    S = torch.view_as_complex(S[:1].cpu().contiguous())
    M = mask.cpu().float().reshape(1, 1, 1, -1)
    H, W = y.shape[-2:]
    L = pics.wavelet_levels(H, W)
    h = torch.tensor(pics.DB4_LO)
    gh = torch.tensor([(-1) ** j for j in range(8)], dtype=torch.float32) * h.flip(0)

    def mats(n):
        k = torch.arange(n // 2)
        lo, hi = torch.zeros(n // 2, n), torch.zeros(n // 2, n)
        for j in range(8):
            lo.index_put_((k, (2 * k + j) % n), h[j].expand(n // 2), accumulate=True)
            hi.index_put_((k, (2 * k + j) % n), gh[j].expand(n // 2), accumulate=True)
        return lo.to(torch.complex64), hi.to(torch.complex64)

    mh = {H >> l: mats(H >> l) for l in range(L)}
    mw = {W >> l: mats(W >> l) for l in range(L)}

    def fft2(v, inv=False):
        v = torch.fft.ifftshift(v, dim=(-2, -1))
        v = (torch.fft.ifft2 if inv else torch.fft.fft2)(v, norm="ortho")
        return torch.fft.fftshift(v, dim=(-2, -1))

    def prox(v, tau):
        c, band = v.clone(), v
        for l in range(L):
            hb, wb = H >> l, W >> l
            (lh_, hh_), (lw, hw) = mh[hb], mw[wb]
            Lx, Hx = band @ lw.T, band @ hw.T
            c[..., :hb // 2, wb // 2:wb], c[..., hb // 2:hb, :wb // 2] = lh_ @ Hx, hh_ @ Lx
            c[..., hb // 2:hb, wb // 2:wb] = hh_ @ Hx
            band = lh_ @ Lx
            c[..., :hb // 2, :wb // 2] = band
        a = c.abs()
        c = torch.where(a > tau, c * ((a - tau) / a.clamp_min(1e-30)), torch.zeros_like(c))
        band = c[..., :H >> L, :W >> L]
        for l in range(L - 1, -1, -1):
            hb, wb = H >> l, W >> l
            (lh_, hh_), (lw, hw) = mh[hb], mw[wb]
            Lx = lh_.T @ band + hh_.T @ c[..., hb // 2:hb, :wb // 2]
            Hx = lh_.T @ c[..., :hb // 2, wb // 2:wb] + hh_.T @ c[..., hb // 2:hb, wb // 2:wb]
            band = Lx @ lw + Hx @ hw
        return band

    alpha = 1.0 / float((S.abs() ** 2).sum(1).amax() * M.abs().amax())
    x = torch.zeros(1, H, W, dtype=torch.complex64)
    z, t = x, 1.0
    t0 = time.perf_counter()
    for _ in range(iters):
        g = (S.conj() * fft2(M * (fft2(S * z[:, None]) - y), inv=True)).sum(1)
        xn = prox(z - alpha * g, alpha * lam)
        tn = (1 + math.sqrt(1 + 4 * t * t)) / 2
        z, x, t = xn + ((t - 1) / tn) * (xn - x), xn, tn
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cpu-iters", type=int, default=ITERS)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_pics.py measures on a CUDA device"
    import mridc_b200 as mb
    from mridc_b200 import pics, synth

    info = card()
    bw = copy_bandwidth()
    rows = []
    for B, C, H, W in GEOMS:
        b = synth.make_batch(B, C, H, W, mask_func=synth.Equispaced1DMask([0.08], [4]), centered=True,
                             normalization="ortho")
        y, S, mask = b["y"].cuda(), b["sensitivity_maps"].cuda(), b["mask"].cuda()
        lam = lam_for(y, S, mask)
        ref = mb.l1_wavelet_recon(y, S, mask, lam, ITERS)  # warm-up
        torch.cuda.synchronize()
        e2e = []
        for _ in range(args.reps):
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            mb.l1_wavelet_recon(y, S, mask, lam, ITERS)
            e.record()
            torch.cuda.synchronize()
            e2e.append(a.elapsed_time(e))
        dc, prox, x = split(y, S, mask, lam)
        assert torch.equal(x, ref), "the split run differs from l1_wavelet_recon"
        ms = sorted(e2e)[len(e2e) // 2]
        pb = prox_bytes(B, H, W, pics.wavelet_levels(H, W))
        cpu_s = cpu_baseline(y, S, mask, lam, args.cpu_iters) * ITERS / args.cpu_iters
        row = {"geometry": "%dx%dx%d" % (C, H, W), "batch": B, "iterations": ITERS, "ms_per_batch": round(ms, 3),
               "slices_per_s": round(1000.0 * B / ms, 2), "e2e_ms_all": [round(v, 3) for v in e2e],
               "dc_ms_per_iter": round(dc, 4), "prox_ms_per_iter": round(prox, 4),
               "prox_share": round(prox / (dc + prox), 4), "prox_bytes_per_iter": pb,
               "prox_GBps": round(pb / (prox * 1e-3) / 1e9, 1), "copy_GBps": round(bw / 1e9, 1),
               "prox_fraction_of_copy_bw": round(pb / (prox * 1e-3) / bw, 3),
               "cpu_fp32_s_per_slice": round(cpu_s, 3), "speedup_vs_cpu": round(cpu_s * 1000.0 * B / ms, 1),
               "card": info}
        print(json.dumps(row), flush=True)
        rows.append(row)
        del y, S, ref, x
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    main()
