#!/usr/bin/env python
"""bench.py -- CIRIM 320x320x15-coil slices/sec (BASELINE.json metric) on N B200s, plus the DC-step HBM GB/s.

    python bench.py --gpus 1 --steps 20 --warmup 3                  # our arm (CUDA, through the public API)
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1  # reference arm: the CPU oracle port
    python bench.py --steps 5 --dump-outputs /tmp/cirim_out         # also write the last step's outputs (.npy)

A "step" = one pass of the hot path (CIRIM.forward: 5 cascades x 8 time steps, ConvGRU, SENSE) over one batch of
`--batch` (default 16) synthetic 15-coil 320x320 slices per GPU, followed by the gather of the reconstructions.  One process
per GPU (torchrun for N > 1), slices sharded across ranks, no data-path collective, weak scaling.
Prints ONE JSON line on rank 0.  Inputs and weights are seeded, so two runs with the same arguments see the same data and
their --dump-outputs files can be compared array for array (e.g. two builds of the library).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

C, H, W = 15, 320, 320
CHW8 = C * H * W * 8
HW8 = H * W * 8
# SURVEY.md section 8(d): algorithmic bytes of one RIM data-consistency gradient per slice (+ mask bytes)
DC_BYTES_PER_SLICE = 2 * CHW8 + HW8 + 2 * HW8
# algorithmic FLOPs of the conv stack per time step per slice (2*MACs), SURVEY 8(d): 19.163 GFLOP
CONV_FLOPS_PER_STEP = 2 * H * W * (4 * 64 * 25 + 2 * (64 * 192 * 2) + 64 * 64 * 9 + 64 * 2 * 9)
# --dump-outputs: complex values kept per intermediate estimate, and at most this many of the final reconstruction (the
# whole volume below that); 40 x 2^16 + 2^22 complex float32 values = 52 MiB at most
DUMP_ESTIMATE_SAMPLES = 1 << 16
DUMP_RECON_MAX = 1 << 22


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


def dc_traffic(B):
    """dram__bytes_read.sum + dram__bytes_write.sum of one DC-gradient launch, from the committed `ncu --set full` capture
    (profiles/*_traffic.json, written by tools/summarise_profiles.py; captured at B = 4 and scaled linearly to B)."""
    import glob

    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")), reverse=True):
        try:
            t = json.load(open(f))["row_dc"]
            return t["dram_bytes_per_launch"] * B / t["slices"]
        except Exception:
            continue
    return None


def conv_traffic(B):
    """DRAM bytes of the regulariser kernels of one time step, from the same committed capture (scaled from B = 4)."""
    import glob

    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")), reverse=True):
        try:
            t = json.load(open(f))["conv_stack"]
            return t["dram_bytes_per_time_step"] * B / t["slices"]
        except Exception:
            continue
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def build_inputs(batch, first_slice=0):
    from mridc_b200 import synth

    return synth.make_batch(batch, C, H, W, centered=False, normalization="backward", first_slice=first_slice)


def cpu_reference_step(sd, cfg, b):
    """The reference's CPU implementation of the path: PyTorch-CPU oracle port of CIRIM.forward."""
    import torch
    from oracle import models as omodels

    with torch.no_grad():
        out = omodels.cirim_forward(sd, cfg, b["y"], b["sensitivity_maps"], b["mask"], None, b["target"])
    return out[-1][-1]


def _seeded_sample(n, k):
    """The same k of n flat positions every run (all n when n <= k), in increasing order."""
    import torch

    return torch.randperm(n, generator=torch.Generator().manual_seed(0))[:k].sort().values


def dump_outputs(path, cascades, volume=None):
    """Write what CIRIM.forward returned in the last timed step as float32 .npy files, complex values as [..., 2] (real,
    imaginary):
      reconstruction.npy    the final estimate cascades[-1][-1] (with N > 1 GPUs the gathered volume), [slices, H, W, 2];
                            above DUMP_RECON_MAX values, a fixed seeded sample of its flat positions, [DUMP_RECON_MAX, 2]
      estimates_sample.npy  every cascade's estimate after every time step at one fixed seeded sample of flat positions,
                            [num_cascades, time_steps, DUMP_ESTIMATE_SAMPLES, 2] (all of them would be 40 volumes); with
                            N > 1 GPUs these are rank 0's slices only, so they cover other slices than a 1-GPU dump"""
    import numpy as np
    import torch

    os.makedirs(path, exist_ok=True)
    rec = torch.view_as_real(cascades[-1][-1] if volume is None else volume)
    if rec.numel() // 2 > DUMP_RECON_MAX:
        rec = rec.reshape(-1, 2)[_seeded_sample(rec.numel() // 2, DUMP_RECON_MAX).to(rec.device)]
    np.save(os.path.join(path, "reconstruction.npy"), rec.float().cpu().numpy())
    idx = _seeded_sample(cascades[0][0].numel(), DUMP_ESTIMATE_SAMPLES).to(rec.device)
    est = torch.stack([torch.stack([torch.view_as_real(e.reshape(-1))[idx] for e in c]) for c in cascades])
    np.save(os.path.join(path, "estimates_sample.npy"), est.float().cpu().numpy())


def run_reference(args):
    import torch
    from mridc_b200 import synth
    import mridc_b200 as mb

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = synth.cirim_cfg("GRU")
    torch.manual_seed(1)
    sd = {k: v.detach().clone() for k, v in mb.CIRIM(cfg).state_dict().items()}
    b = build_inputs(1)
    for _ in range(args.warmup):
        cpu_reference_step(sd, cfg, b)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_reference_step(sd, cfg, b)
    dt = time.perf_counter() - t0
    val = args.steps / dt
    sample = "%d step(s) of 1 slice each (full CIRIM 5x8 GRU, 15x320x320), %d warm-up, torch-CPU %d threads" % (
        args.steps, args.warmup, cores)
    line = {
        "impl": "reference", "metric": "cirim_320x320x15coil_slices_per_sec", "value": val, "unit": "slices/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the repo arm's own config (the metric is per slice; a CPU step is a bounded sample of that workload: one slice)
        "config": workload_config(args.batch, args.gpus),
        "cpu_baseline": {"value": val, "unit": "slices/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "slices/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def workload_config(batch, n_gpus):
    return {"workload": "CIRIM 5 cascades x 8 time steps, ConvGRU 64 filters (k5/k3d2/k3), SENSE, no_dc, keep_eta, "
                        "fft non-centered/backward; 15-coil 320x320 knee-shaped slices, 4x equispaced 1-D mask "
                        "(BASELINE.json configs[2])",
            "slices_per_gpu_per_step": batch, "global_slices_per_step": batch * n_gpus,
            "parallelism": "slice-sharded x%d, gather of reconstructions only" % n_gpus,
            "l2": "per-step working set (y+S %.0f MB, hidden states %.0f MB) exceeds the 126 MB L2; no flush needed"
                  % (batch * 2 * CHW8 / 1e6, batch * 4 * 64 * H * W * 4 / 1e6)}


def run_extras(model, d, dev, e0, e1):
    """Secondary, driver-visible measurements (rank 0, N = 1): single-slice latency (the reference ships batch_size 1,
    base_cirim_run.yaml:71), E2EVN (BASELINE.json configs[1]) and the brain geometry of configs[3] on one GPU."""
    import numpy as np
    import torch
    import mridc_b200 as mb
    from mridc_b200 import _ops, synth

    def timed(fn, n, w=3):
        for _ in range(w):
            fn()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    out = {}
    # ---- B = 1 latency through CIRIM.forward (inputs resident; the time loop of each cascade replays a CUDA graph) ----
    one = {k: (d[k][:1].contiguous() if d[k].shape[0] > 1 else d[k]) for k in ("y", "sensitivity_maps", "mask", "target")}

    def fwd1():
        return next(model(one["y"], one["sensitivity_maps"], one["mask"], None, one["target"]))[-1][-1]

    lat = timed(fwd1, 20, 5)
    eng = model.cirim[0]._tc_engine
    kern = None
    if eng:
        step1, _ = eng.bench_step(1, H, W, dev)
        mcan = _ops.canonical_mask(one["mask"], 1, H, W)[0]
        yh1 = _ops.dc_hybrid_prepare(one["y"], mcan, False)
        eta1 = torch.randn((1, H, W, 2), device=dev)
        g41 = torch.empty((1, H, W, 4), device=dev)
        dc1 = timed(lambda: _ops.dc_rim_grad(eta1, one["y"], one["sensitivity_maps"], mcan, 1.0, False, "backward", out=g41,
                                             nhwc=True, y_hybrid=yh1), 40)
        kern = 40 * (timed(step1, 20) + dc1)
    out["latency_b1"] = {"ms": lat, "kernel_ms": kern, "ratio": (lat / kern) if kern else None,
                         "note": "CIRIM.forward on ONE slice, inputs resident; kernel_ms = 40 x (conv stack + DC gradient) "
                                 "timed back to back at B = 1"}
    # ---- E2EVN, configs[1] ----
    Bv = 8
    np.random.seed(123)
    dv = synth.make_batch(Bv, C, H, W, mask_func=synth.Gaussian1DMask([0.7], [4]), seed=123, mask_dtype="uint8")
    torch.manual_seed(1)
    vn = mb.VarNet(synth.varnet_cfg()).eval().to(dev)
    hv = {k: dv[k].pin_memory() for k in ("y", "sensitivity_maps", "mask", "target")}
    gv = {k: v.to(dev) for k, v in hv.items()}
    ms = timed(lambda: vn(gv["y"], gv["sensitivity_maps"], gv["mask"], None, gv["target"]), 8)

    def vn_e2e():
        t = {k: v.to(dev, non_blocking=True) for k, v in hv.items()}
        return vn(t["y"], t["sensitivity_maps"], t["mask"], None, t["target"]).cpu()

    ms_e = timed(vn_e2e, 8)
    wsv = torch.empty((2, Bv, C, H, W, 2), device=dev)
    img = torch.randn(Bv, H, W, 2, device=dev)
    dcw = torch.ones(1, device=dev)
    o5 = torch.empty_like(gv["y"])

    def dc_block():
        _ops.sens_reduce(gv["y"], gv["sensitivity_maps"], False, "backward", ws=wsv)
        _ops.sens_expand_softdc(img, gv["sensitivity_maps"], gv["y"], gv["y"], gv["y"], gv["mask"], dcw, False, False,
                                "backward", out=o5, ws=wsv)

    ms_dc = timed(dc_block, 20)
    dcb = Bv * (6 * CHW8 + 2 * HW8)
    peaks = load_peaks()
    out["e2evn"] = {"metric": "e2evn_320x320x15coil_slices_per_sec", "value": Bv / ms * 1e3,
                    "e2e": Bv / ms_e * 1e3, "unit": "slices/s", "slices_per_step": Bv,
                    "workload": "E2EVN 12 cascades, U-Net 14 ch / 2 pools, 15x320x320, 4x Gaussian 1-D (BASELINE.json configs[1])",
                    "soft_dc_block": {"ms": ms_dc, "algorithmic_bytes": dcb, "achieved_gbs": dcb / ms_dc / 1e6,
                                      "frac": dcb / ms_dc / 1e6 / peaks["hbm_gbs"], "share_of_step": 12 * ms_dc / ms}}
    del vn, gv, wsv, o5
    # ---- configs[3]: CIRIM on 16-coil 640x320 brain-shaped slices, 8x equispaced mask (one GPU's share) ----
    Bb, Cb, Hb = 8, 16, 640
    db = synth.make_batch(Bb, Cb, Hb, W, mask_func=synth.Equispaced1DMask([0.04], [8]))
    gb = {k: db[k].to(dev) for k in ("y", "sensitivity_maps", "mask", "target")}
    msb = timed(lambda: next(model(gb["y"], gb["sensitivity_maps"], gb["mask"], None, gb["target"]))[-1][-1], 5, 2)
    mcb = _ops.canonical_mask(gb["mask"], Bb, Hb, W)[0]
    yhb = _ops.dc_hybrid_prepare(gb["y"], mcb, False)
    etab = torch.randn((Bb, Hb, W, 2), device=dev)
    g4b = torch.empty((Bb, Hb, W, 4), device=dev)
    dcb_ms = timed(lambda: _ops.dc_rim_grad(etab, gb["y"], gb["sensitivity_maps"], mcb, 1.0, False, "backward", out=g4b,
                                            nhwc=True, y_hybrid=yhb), 40)
    bytes_b = Bb * (2 * Cb * Hb * W * 8 + 3 * Hb * W * 8) + W
    out["brain_cirim"] = {"metric": "cirim_640x320x16coil_slices_per_sec", "value": Bb / msb * 1e3, "unit": "slices/s",
                          "slices_per_step": Bb,
                          "workload": "CIRIM 5x8 ConvGRU, 16-coil 640x320 brain-shaped slices, 8x equispaced mask "
                                      "(BASELINE.json configs[3], one GPU's share of the batch)",
                          "dc_gradient": {"ms": dcb_ms, "algorithmic_bytes": bytes_b, "achieved_gbs": bytes_b / dcb_ms / 1e6,
                                          "frac": bytes_b / dcb_ms / 1e6 / peaks["hbm_gbs"]}}
    # ---- configs[3]: E2EVN on the same brain-shaped slices ----
    torch.manual_seed(1)
    vnb = mb.VarNet(synth.varnet_cfg()).eval().to(dev)
    msvb = timed(lambda: vnb(gb["y"], gb["sensitivity_maps"], gb["mask"], None, gb["target"]), 5, 2)
    out["brain_e2evn"] = {"metric": "e2evn_640x320x16coil_slices_per_sec", "value": Bb / msvb * 1e3, "unit": "slices/s",
                          "slices_per_step": Bb,
                          "workload": "E2EVN 12 cascades, 16-coil 640x320 brain-shaped slices, 8x equispaced mask "
                                      "(BASELINE.json configs[3], one GPU's share of the batch)"}
    del vnb, gb
    # ---- the IndRNN variant of the headline network (the cell base_cirim_run.yaml ships) ----
    torch.manual_seed(1)
    mi = mb.CIRIM(synth.cirim_cfg("IndRNN")).eval().to(dev)
    Bi = min(16, d["y"].shape[0])
    di = {k: (d[k][:Bi].contiguous() if d[k].shape[0] > 1 else d[k]) for k in ("y", "sensitivity_maps", "mask", "target")}
    msi = timed(lambda: next(mi(di["y"], di["sensitivity_maps"], di["mask"], None, di["target"]))[-1][-1], 5, 2)
    out["cirim_indrnn"] = {"metric": "cirim_indrnn_320x320x15coil_slices_per_sec", "value": Bi / msi * 1e3, "unit": "slices/s",
                           "slices_per_step": Bi,
                           "workload": "CIRIM 5x8 with IndRNN cells (base_cirim_run.yaml), 15x320x320, same inputs as the "
                                       "headline"}
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    import mridc_b200 as mb
    from mridc_b200 import _lib, _ops, sharding, synth

    B = args.batch
    cfg = synth.cirim_cfg("GRU")
    torch.manual_seed(1)
    model = mb.CIRIM(cfg).eval()
    sd_cpu = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model = model.to(dev)
    host = build_inputs(B, first_slice=rank * B)
    pinned = {k: host[k].pin_memory() for k in ("y", "sensitivity_maps", "mask", "target")}
    d = {k: v.to(dev) for k, v in pinned.items()}
    n_global = B * world

    pending = []
    kept = {}

    def step_resident(keep=False):
        out = next(model(d["y"], d["sensitivity_maps"], d["mask"], None, d["target"]))
        if keep:
            kept["out"] = out  # every estimate of this step, for --dump-outputs
        rec = out[-1][-1]
        if world == 1:
            return rec
        # only rank 0 needs the volume (the reference's test_epoch_end): point-to-point gather on NCCL's own stream,
        # waited for one step later so that it overlaps with the next step's kernels
        if pending:
            pending.pop().wait()
        pending.append(sharding.gather_reconstructions(rec, n_global, dst=0, async_op=True))
        return rec

    def drain():
        return pending.pop().wait() if pending else None

    def barrier_sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- the DC gradient kernel timed ALONE, before the long loop heats the part into its power cap (rank 0): the kernel
    # is issue / latency bound, so its time follows the SM clock; the contract figure below (roofline_dc.frac) is the one
    # measured after the timed region, at the clocks of the sustained run
    dc_alone_ms = None
    if rank == 0 and W == 320 and C <= 16:
        _eta = d["y"].new_zeros((B, H, W, 2)).normal_()
        _mcan = _ops.canonical_mask(d["mask"], B, H, W)[0]
        _yh = _ops.dc_hybrid_prepare(d["y"], _mcan, False)
        _g8 = torch.zeros(_lib.load().mrb_g8_bytes(B, H, W), dtype=torch.uint8, device=dev)
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(5):
            _ops.dc_rim_grad(_eta, d["y"], d["sensitivity_maps"], _mcan, 1.0, False, "backward", out=_g8, nhwc=2, y_hybrid=_yh)
        torch.cuda.synchronize()
        ea.record()
        for _ in range(40):
            _ops.dc_rim_grad(_eta, d["y"], d["sensitivity_maps"], _mcan, 1.0, False, "backward", out=_g8, nhwc=2, y_hybrid=_yh)
        eb.record()
        torch.cuda.synchronize()
        dc_alone_ms = ea.elapsed_time(eb) / 40
        del _eta, _yh, _g8
    # ---- device-resident timing --------------------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        step_resident()
    if world > 1:
        # outside the timed region: what rank 0 gathered must equal, bit for bit, what each rank computed locally
        full = drain()
        local_rec = step_resident()
        drain()
        lr = torch.view_as_real(local_rec).contiguous()  # NCCL has no complex type
        mine = [torch.zeros_like(lr) for _ in range(world)] if rank == 0 else None
        dist.gather(lr, mine, dst=0)
        if rank == 0:
            assert full is not None and torch.equal(torch.view_as_real(full), torch.cat(mine, 0)), \
                "gathered volume != per-rank results"
    barrier_sync()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    _lib.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        step_resident(keep=args.dump_outputs is not None and rank == 0 and i == args.steps - 1)
    gathered = drain()
    e1.record()
    barrier_sync()
    launches = _lib.launch_count()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = ms.item()
    clocks = sampler.stop() if sampler else None
    if kept:
        dump_outputs(args.dump_outputs, kept.pop("out"), gathered)

    # ---- end-to-end timing: host buffers, H2D + compute + D2H of the reconstruction every step ------
    out_host = torch.empty((B, H, W), dtype=torch.complex64).pin_memory()

    from mridc_b200.pipeline import HostPrefetcher

    def run_e2e(n):
        # the public streaming path: pinned host batches -> HostPrefetcher (upload of batch k+1 on a copy stream while
        # batch k is reconstructed) -> model -> reconstruction copied back to pinned host memory, every step
        feed = ({k: pinned[k] for k in ("y", "sensitivity_maps", "mask")} for _ in range(n))
        for bt in HostPrefetcher(feed, dev):
            out = next(model(bt["y"], bt["sensitivity_maps"], bt["mask"], None, d["target"]))
            rec = out[-1][-1]
            if world > 1:
                full = sharding.gather_reconstructions(rec, n_global, dst=0)
                rec = full[:B] if rank == 0 else rec
            out_host.copy_(rec, non_blocking=True)

    run_e2e(2)
    barrier_sync()
    e0.record()
    run_e2e(args.steps)
    e1.record()
    barrier_sync()
    ms2 = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_val = n_global * args.steps / (ms2.item() / 1e3)
    h2d = sum(pinned[k].numel() * pinned[k].element_size() for k in ("y", "sensitivity_maps", "mask"))
    d2h = out_host.numel() * out_host.element_size()

    # ---- per-kernel roofline passes (rank 0): CUDA events on the launching stream ---------------------
    roof, roof_conv, share = None, None, None
    if rank == 0:
        peaks = load_peaks()
        eta = d["y"].new_zeros((B, H, W, 2)).normal_()
        ws = torch.empty((2, B, C, H, W, 2), device=dev)
        outg = torch.empty((B, 4, H, W), device=dev)
        mcan = _ops.canonical_mask(d["mask"], B, H, W)[0]
        n_it = 40
        # the product path: hybrid-space row form (1-D mask), hybrid k-space prepared once per slice batch
        yhyb = _ops.dc_hybrid_prepare(d["y"], mcan, False, ws=ws[0])
        # the form the time loop launches at W = 320: G8 output (the regulariser's split-bf16 conv input with its
        # replicate border, 16 B per position like the fp32 channels-last form)
        use_g8 = W == 320 and C <= 16
        outg4 = (torch.zeros(_lib.load().mrb_g8_bytes(B, H, W), dtype=torch.uint8, device=dev) if use_g8
                 else torch.empty((B, H, W, 4), device=dev))

        def dc_call():
            _ops.dc_rim_grad(eta, d["y"], d["sensitivity_maps"], mcan, 1.0, False, "backward", out=outg4,
                             nhwc=2 if use_g8 else True, y_hybrid=yhyb)

        # the general three-pass operator is what 2-D masks (Gaussian2D / Poisson2D / Equispaced2D) take: time it on one
        m2d = (torch.rand((1, H, W), device=dev) < 0.25).to(torch.uint8)

        def dc_call_3pass():
            _ops.dc_rim_grad(eta, d["y"], d["sensitivity_maps"], m2d, 1.0, False, "backward", out=outg, ws=ws)

        def time_it(fn):
            for _ in range(5):
                fn()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(n_it):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n_it

        dc_ms = time_it(dc_call)
        dc3_ms = time_it(dc_call_3pass)
        dc_bytes = B * DC_BYTES_PER_SLICE + mcan.numel() * mcan.element_size()
        dc_gbs = dc_bytes / (dc_ms * 1e-3) / 1e9
        roof_dc = {"bound": "hbm",
                   "kernel": "DC gradient, hybrid-space row form (row_dc320_kernel: S*eta -> FFT_W -> mask*(. - yh) -> IFFT_W "
                             "-> sum_c conj(S)*., register-resident 16x20 transforms, hybrid k-space rows staged by bulk "
                             "copies, G8 output; the H transforms cancel for 1-D masks, yh prepared once per batch)",
                   "achieved": dc_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": dc_gbs / peaks["hbm_gbs"],
                   "frac_of_nominal_8000": dc_gbs / 8000.0, "traffic": dc_traffic(B), "peak_src": peaks["src"],
                   "ms_per_launch_group": dc_ms, "algorithmic_bytes": dc_bytes,
                   "general_three_pass_ms": dc3_ms, "general_three_pass_gbs": dc_bytes / (dc3_ms * 1e-3) / 1e9,
                   "timed_alone_ms": dc_alone_ms,
                   "timed_alone_frac": (dc_bytes / (dc_alone_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]) if dc_alone_ms else None,
                   "note": "algorithmic bytes = SURVEY 8(d) contract figure (S and y once, eta in, 4-channel out); the row "
                           "form actually reads S once and only the sampled columns of yh.  ms_per_launch_group / frac: 40 "
                           "launches right after the timed region (clocks of the power-capped sustained run); "
                           "timed_alone_*: the same 40 launches before the first step (boost clocks); general_three_pass_*: "
                           "the operator every 2-D mask takes, timed on a random 2-D mask of density 0.25"}
        # conv stack of one time step (the compute-dominant kernels), tensor-core channels-last engine
        blk = model.cirim[0]
        eng = blk._tc_engine
        etab = eta.clone()
        if eng:
            conv_stack, kname = eng.bench_step(B, H, W, dev)
            note = ("error-compensated split-bf16 products on tcgen05 (a_hi*b_hi + a_hi*b_lo + a_lo*b_hi, fp32 accumulation in "
                    "TMEM): 3 bf16 MMAs per product; achieved counts the algorithmic fp32 FLOPs once")
        else:
            g4n = torch.randn((B, 4, H, W), device=dev)
            hn = [torch.randn((B, 64, H, W), device=dev) * 0.1 for _ in range(2)]

            def conv_stack():
                x = g4n
                for hi_, layer in enumerate(blk.layers):
                    x = layer(x, hn[hi_])
                return blk.final_layer[0](x, residual_nhwc=etab)
            kname = "fp32 CUDA-core ConvGRU stack of one time step"
            note = "exact-fp32 CUDA-core path (FFMA)"
        for _ in range(3):
            conv_stack()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(10):
            conv_stack()
        e1.record()
        torch.cuda.synchronize()
        cv_ms = e0.elapsed_time(e1) / 10
        tf = B * CONV_FLOPS_PER_STEP / (cv_ms * 1e-3) / 1e12
        roof_conv = {"bound": "tensor", "kernel": kname, "achieved": tf, "peak": peaks["bf16_tflops_sustained"],
                     "unit": "TFLOP/s", "frac": tf / peaks["bf16_tflops_sustained"], "traffic": conv_traffic(B),
                     "peak_src": peaks["src"], "ms_per_time_step": cv_ms, "note": note,
                     # an fp32-grade result costs 3 bf16 products per MAC: the same time expressed against that
                     # ceiling (peak / 3)
                     "frac_of_split_bf16_ceiling": (3.0 * tf / peaks["bf16_tflops_sustained"]) if eng else None}
        step_ms = ms_total / args.steps
        share = {"dc_share_of_step": 40 * dc_ms / step_ms, "conv_share_of_step": 40 * cv_ms / step_ms}
        roof = roof_conv if cv_ms > dc_ms else roof_dc
        roof = dict(roof)
        extra = {"roofline_dc": roof_dc, "roofline_conv": roof_conv, "kernel_shares": share}
    if rank == 0 and world == 1 and not args.no_extras:
        extra["extras"] = run_extras(model, d, dev, e0, e1)
    # ---- CPU baseline (rank 0, N = 1 only): bounded sample of the same workload ------------------------
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        one = {k: host[k][:1] if host[k].shape[0] == B else host[k] for k in ("y", "sensitivity_maps", "mask", "target")}
        cpu_reference_step(sd_cpu, cfg, one)  # warm-up (thread pool, allocator, oneDNN primitives)
        t0 = time.perf_counter()
        ref = cpu_reference_step(sd_cpu, cfg, one)
        dt = time.perf_counter() - t0
        ours = next(model(d["y"][:1], d["sensitivity_maps"][:1], d["mask"], None, d["target"][:1]))[-1][-1]
        a = torch.view_as_real(ours.cpu()).double()
        b = torch.view_as_real(ref).double()
        cpu_base = {"value": 1.0 / dt, "unit": "slices/s", "cores": cores, "kind": "port",
                    "sample": "1 slice of the same workload (full CIRIM 5x8), after 1 warm-up slice, torch-CPU %d threads, %.1f s"
                              % (cores, dt),
                    "parity_rel_l2_vs_cuda": ((a - b).norm() / b.norm()).item()}
    if rank == 0:
        val = n_global * args.steps / (ms_total / 1e3)
        line = {
            "metric": "cirim_320x320x15coil_slices_per_sec", "value": val, "unit": "slices/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(B, world), "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": e2e_val, "unit": "slices/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "roofline": roof, "cpu_baseline": cpu_base,
        }
        line.update(extra)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="slices per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary measurements (latency, E2EVN, brain)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA arm (--impl ours)")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
