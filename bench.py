#!/usr/bin/env python
"""bench.py -- headline benchmark of the motion-compensation hot path (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--frames F] [--dump-outputs DIR]

One "step" = one pass of the soft-mode (softmax) forward splat over one batch of F synthetic
1080p fp32 frames (BASELINE.json north_star: "fp32 softmax-splat forward on 1080p frames"; the
frames are C1/C3-shaped: 3 x 1080 x 1920, smooth synthetic flow of ~8 px). Prints ONE JSON line.

  value        whole-job Mpixel/s (source pixels, not x C), inputs resident in HBM, CUDA events,
               max over ranks; weak scaling (every rank owns its own F frames, no collective)
  e2e          same metric through the public Python API from PINNED HOST buffers: H2D of the
               step's inputs, the op, D2H of the result, all inside the timed region
  roofline     algorithmic bytes (36 B/px, SURVEY.md section 8d) / measured duration of one
               frame's launch pair (k_splat_step scatters frame k into the L2-resident accumulator
               slot, k_splat_epilogue normalises it; 2F launches per step of F frames) vs the
               measured HBM copy peak
  cpu_baseline the oracle port (C + pthreads over frames) on a bounded sample, rank 0, N=1 only
  extra        secondary configs of BASELINE.json (C1 avg latency, C2 bf16 latents, C3 residual
               recipe + backwarp, C4 fwd+bwd), measured outside the timed region

--impl reference times the reference's path on the host cores. The reference has NO CPU
implementation (controlnet/softsplat.py:347-348 asserts) and CuPy is not installed, so this arm
runs the committed CPU port of its kernel (oracle/, kind "port") with all host threads.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H, W, C = 1080, 1920, 3
ALG_BYTES_PER_PX = (2 * C + 3) * 4          # soft fwd: read C in + 1 metric + 2 flow, write C out (fp32)


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def _smooth_flow(torch, n, h, w, amp, device, gen):
    """~RAFT-like flow: low-resolution noise upsampled bilinearly, amplitude ~amp px."""
    low = torch.randn(n, 2, max(h // 32, 2), max(w // 32, 2), device=device, generator=gen)
    return torch.nn.functional.interpolate(low, size=(h, w), mode="bicubic", align_corners=False) * amp


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            p = [x.strip() for x in line.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


WORKLOAD = ("soft (softmax) forward splat, fp32, {F}x3x1080x1920 frames per GPU per step, synthetic flow ~8 px "
            "(bicubic-upsampled noise, mean |dflow/dx| 0.28 px/px: rougher than real optical flow; extra.headline_on_smooth_flow has 0.03)")


def _config(frames):
    """The SAME dict in both arms (the driver compares them)."""
    return {"workload": WORKLOAD.format(F=frames), "frames_per_gpu": frames,
            "l2_policy": f"inputs+outputs per step = {(36 * frames * H * W) >> 20} MiB per GPU, larger than the 126 MB L2; no flush needed",
            "partition": "frames sharded by rank, no data-path collective"}


_cpu_inputs = {}


def _cpu_port_mpixel_s(frames, threads, repeats=1):
    """Soft-mode forward on the host: the oracle's C kernel (frame-parallel pthreads) + the mode
    wrapper's pre/post ops in torch CPU, exactly the reference composition (softsplat.py:246-270).
    The synthetic inputs are generated once per frame count (untimed)."""
    import torch
    from oracle import oracle as orc

    torch.set_num_threads(max(1, threads))      # torchrun exports OMP_NUM_THREADS=1: give the pre/post ops the cores too
    if frames not in _cpu_inputs:
        torch.manual_seed(0)
        _cpu_inputs.clear()
        _cpu_inputs[frames] = (torch.rand(frames, C, H, W), -torch.rand(frames, 1, H, W), _smooth_flow(torch, frames, H, W, 8.0, "cpu", None))
    tin, metric, flow = _cpu_inputs[frames]
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        e = metric.exp()
        x = torch.cat([tin * e, e], 1)
        s = torch.from_numpy(orc.splat_fwd_mt(x.numpy(), flow.numpy(), threads))
        out = s[:, :-1] / (s[:, -1:] + 0.0000001)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    assert out.shape == tin.shape
    return frames * H * W / best / 1e6, best


def run_reference(args):
    """Reference arm: the path on host cores (see module docstring for why it is a port)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    threads = orc.max_threads()
    frames = max(4, (args.frames // max(threads, 1)) * threads) if args.frames >= threads else args.frames   # whole rounds of the thread pool
    for _ in range(min(args.warmup, 1)):
        _cpu_port_mpixel_s(frames, threads)
    t0 = time.perf_counter()
    vals = [_cpu_port_mpixel_s(frames, threads)[0] for _ in range(args.steps)]
    dt = time.perf_counter() - t0
    v = statistics.median(vals)
    sample = f"{frames} synthetic 1080p frames per step, soft fwd fp32 (C kernel over {threads} pthreads + torch CPU pre/post ops)"
    print(json.dumps({
        "impl": "reference", "metric": "softsplat soft-mode forward throughput, 1080p fp32 frames", "value": round(v, 2),
        "unit": "Mpixel/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dt / max(args.steps, 1) * 1e3, 2), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config(args.frames),
        "cpu_baseline": {"value": round(v, 2), "unit": "Mpixel/s", "cores": threads, "kind": "port",
                         "sample": sample + f"; each step = {frames} of the workload's frames on rank 0's host cores"},
        "e2e": {"value": round(v, 2), "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference has no CPU path and CuPy is absent: this is the committed CPU port of its kernel (oracle/)",
    }))


def _time_cuda(torch, fn, iters, warm=3):
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters          # ms


def _extras(torch, d, dev, gen, peak):
    """Secondary BASELINE.json configs; each a few hundred ms. Never part of the timed region."""
    ex = {}
    try:
        # the headline workload again on flow as smooth as real optical flow (same ~8 px amplitude, noise cell
        # 256 px instead of 32 px): register merging then removes most L2 reduction sectors
        F2 = 32
        t_ = torch.rand(F2, 3, H, W, device=dev, generator=gen); m_ = -torch.rand(F2, 1, H, W, device=dev, generator=gen)
        low = torch.randn(F2, 2, 4, 7, device=dev, generator=gen)
        fs = torch.nn.functional.interpolate(low, size=(H, W), mode="bicubic", align_corners=False) * 8.0
        ms = _time_cuda(torch, lambda: d.softsplat(t_, fs, m_, "soft"), 5, 3)
        ex["headline_on_smooth_flow_32x3x1080x1920_f32"] = {
            "mean_abs_dflow_dx": round(float((fs[:, :, :, 1:] - fs[:, :, :, :-1]).abs().mean()), 4), "us_per_frame": round(ms * 1e3 / F2, 2),
            "mpixel_s": round(F2 * H * W / ms / 1e3, 1), "alg_gbs": round(36 * F2 * H * W / ms / 1e6, 1),
            "frac_of_peak": round(36 * F2 * H * W / ms / 1e6 / peak, 3)}
        # BASELINE.md's wording read literally: gaussian_blur(randn * 8 px, sigma = 16 px), no re-scaling
        # (sub-pixel, very coherent motion)
        k = torch.arange(-48, 49, device=dev, dtype=torch.float32)
        k = torch.exp(-0.5 * (k / 16.0) ** 2); k = (k / k.sum()).view(1, 1, 1, -1)
        fl_ = torch.randn(F2 * 2, 1, H, W, device=dev, generator=gen) * 8.0
        fl_ = torch.nn.functional.conv2d(torch.nn.functional.pad(fl_, (48, 48, 0, 0), mode="replicate"), k)
        fl_ = torch.nn.functional.conv2d(torch.nn.functional.pad(fl_, (0, 0, 48, 48), mode="replicate"), k.transpose(2, 3))
        fl_ = fl_.view(F2, 2, H, W).contiguous()
        ms = _time_cuda(torch, lambda: d.softsplat(t_, fl_, m_, "soft"), 5, 3)
        ex["headline_on_literal_blurred_flow_32x3x1080x1920_f32"] = {
            "flow_std_px": round(float(fl_.std()), 3), "us_per_frame": round(ms * 1e3 / F2, 2), "mpixel_s": round(F2 * H * W / ms / 1e3, 1),
            "frac_of_peak": round(36 * F2 * H * W / ms / 1e6 / peak, 3)}
        del t_, m_, fs, low, fl_
        # C1: avg forward of single 1x3x1080x1920 frames, rotating pool of 16 distinct frames (> L2)
        pool = [(torch.rand(1, 3, H, W, device=dev, generator=gen), _smooth_flow(torch, 1, H, W, 8.0, dev, gen)) for _ in range(16)]
        it = [0]
        def c1():
            t, f = pool[it[0] % 16]; it[0] += 1
            d.softsplat(t, f, None, "avg")
        ms = _time_cuda(torch, c1, 64, 16)
        ex["C1_avg_fwd_1x3x1080x1920_f32"] = {"us_per_call": round(ms * 1e3, 2), "mpixel_s": round(H * W / ms / 1e3, 1),
                                              "alg_gbs": round(32 * H * W / ms / 1e6, 1), "frac_of_peak": round(32 * H * W / ms / 1e6 / peak, 3)}
        del pool
        # C2: soft forward of SD latents 4x4x135x240 bf16 (launch-latency bound): us per call
        lat = (torch.randn(4, 4, 135, 240, device=dev, generator=gen) * 0.18215).bfloat16()
        met = (-torch.randn(4, 1, 135, 240, device=dev, generator=gen).abs()).bfloat16()
        fl = torch.randn(4, 2, 135, 240, device=dev, generator=gen)
        flb = fl.bfloat16()
        ms = _time_cuda(torch, lambda: d.softsplat(lat, flb, met, "soft"), 200, 20)
        ms32 = _time_cuda(torch, lambda: d.softsplat(lat, fl, met, "soft"), 200, 20)
        # the same call replayed from a CUDA graph: device time without the Python/ctypes host path
        gs = torch.cuda.Stream(); gs.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(gs):
            d.softsplat(lat, flb, met, "soft")
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr, stream=gs):
                d.softsplat(lat, flb, met, "soft")
        torch.cuda.synchronize()
        msg = _time_cuda(torch, gr.replay, 200, 20)
        l0 = d.launch_count(); d.softsplat(lat, flb, met, "soft"); c2_launches = d.launch_count() - l0
        ex["C2_soft_fwd_4x4x135x240_bf16"] = {"us_per_call": round(ms * 1e3, 2), "us_per_call_fp32_flow": round(ms32 * 1e3, 2),
                                              "us_per_call_cuda_graph": round(msg * 1e3, 2), "launches_per_call": c2_launches,
                                              "mpixel_s": round(4 * 135 * 240 / ms / 1e3, 1)}
        # the live consumer: the 16 splats of one DualFlowControlNet forward (extractors.py:280-314), batch 2
        pyr = []
        for ch, r in ((160, 64), (160, 32), (320, 16), (640, 8)):
            feat = torch.randn(2, ch, r, r, device=dev, generator=gen); f_ = torch.randn(2, 2, r, r, device=dev, generator=gen) * 0.3
            m_ = torch.randn(2, 1, r, r, device=dev, generator=gen) * 0.1
            pyr.append((feat, f_, -f_, m_))
        def pyramid():
            for feat, ff, fb, m_ in pyr:
                of = d.compute_mask(ff, fb); ob = d.compute_mask(fb, ff)
                d.softsplat(feat, ff, m_, "soft"); d.softsplat(feat, fb, m_, "soft")
        with torch.no_grad():
            msp = _time_cuda(torch, pyramid, 50, 10)
        ex["controlnet_pyramid_16_splats_batch2_f32"] = {"us_per_forward": round(msp * 1e3, 1), "us_per_splat": round(msp * 1e3 / 16, 2)}
        # the same 16 splats + the 4 fusions as FOUR fused calls (dcb_bidir_block_fwd: one library call per scale, learned-metric stand-in)
        def pyramid_fused():
            for feat, ff, fb, m_ in pyr:
                d.bidirectional_block(feat, feat, ff, fb, m_, m_)
        with torch.no_grad():
            msf = _time_cuda(torch, pyramid_fused, 50, 10)
        ex["controlnet_pyramid_4_fused_blocks_batch2_f32"] = {"us_per_forward": round(msf * 1e3, 1), "includes": "16 splats + 4 confidence fusions with hole fill"}
        # ... and as ONE call for the whole pyramid (dcb_bidir_pyramid_fwd: two launches + one memset for all four scales)
        levels = [(feat, feat, ff, fb, m_, m_) for feat, ff, fb, m_ in pyr]
        with torch.no_grad():
            ms1 = _time_cuda(torch, lambda: d.bidirectional_pyramid(levels), 50, 10)
            l0 = d.launch_count(); d.bidirectional_pyramid(levels); per = d.launch_count() - l0
            gs = torch.cuda.Stream(); gs.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(gs):
                d.bidirectional_pyramid(levels)
                gp = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gp, stream=gs):
                    d.bidirectional_pyramid(levels)
            torch.cuda.synchronize()
            msgp = _time_cuda(torch, gp.replay, 100, 10)
        ex["controlnet_pyramid_one_call_batch2_f32"] = {"us_per_forward": round(ms1 * 1e3, 1), "us_per_forward_cuda_graph": round(msgp * 1e3, 1),
                                                        "kernel_launches": per, "includes": "16 splats + 4 confidence fusions with hole fill"}
        # C3: 64-frame 1080p warp + residual: fused splat recipe and backwarp + residual
        n3 = 64
        img = torch.rand(n3, 3, H, W, device=dev, generator=gen); gt = torch.rand(n3, 3, H, W, device=dev, generator=gen)
        f1 = _smooth_flow(torch, n3, H, W, 8.0, dev, gen); f2 = -f1 + 0.5 * _smooth_flow(torch, n3, H, W, 1.0, dev, gen)
        ms = _time_cuda(torch, lambda: d.residual_conditioning(img, f1, f2, gt, "dataset"), 5, 2)
        ex["C3_residual_recipe_64x3x1080x1920_f32"] = {"ms": round(ms, 3), "mpixel_s": round(n3 * H * W / ms / 1e3, 1),
                                                       "alg_gbs": round(64 * n3 * H * W / ms / 1e6, 1), "frac_of_peak": round(64 * n3 * H * W / ms / 1e6 / peak, 3)}
        ms = _time_cuda(torch, lambda: d.backwarp_residual(img, f1, gt), 5, 2)
        ex["C3_backwarp_residual_64x3x1080x1920_f32"] = {"ms": round(ms, 3), "mpixel_s": round(n3 * H * W / ms / 1e3, 1),
                                                         "alg_gbs": round(56 * n3 * H * W / ms / 1e6, 1), "frac_of_peak": round(56 * n3 * H * W / ms / 1e6 / peak, 3)}
        del img, gt, f1, f2
        # forward + backward (all three gradients) on the headline's frames: (6C+10)*4 = 112 B/px
        nb = 16
        ti = torch.rand(nb, 3, H, W, device=dev, generator=gen).requires_grad_(True)
        me = (-torch.rand(nb, 1, H, W, device=dev, generator=gen)).requires_grad_(True)
        fl = _smooth_flow(torch, nb, H, W, 8.0, dev, gen).requires_grad_(True)
        go = torch.randn(nb, 3, H, W, device=dev, generator=gen)
        def fb():
            ti.grad = me.grad = fl.grad = None
            d.softsplat(ti, fl, me, "soft").backward(go)
        ms = _time_cuda(torch, fb, 5, 2)
        ex["headline_fwd_bwd_16x3x1080x1920_f32"] = {"us_per_frame": round(ms * 1e3 / nb, 1), "mpixel_s": round(nb * H * W / ms / 1e3, 1),
                                                      "alg_gbs": round(112 * nb * H * W / ms / 1e6, 1),
                                                      "frac_of_peak": round(112 * nb * H * W / ms / 1e6 / peak, 3)}
        del ti, me, fl, go
        # C4: soft forward + backward on 8x64x256x256 fp32 (ControlNet training shape), all grads
        ti = torch.randn(8, 64, 256, 256, device=dev, generator=gen).requires_grad_(True)
        me = (torch.randn(8, 1, 256, 256, device=dev, generator=gen) * 0.5).requires_grad_(True)
        fl = _smooth_flow(torch, 8, 256, 256, 4.0, dev, gen).requires_grad_(True)
        go = torch.randn(8, 64, 256, 256, device=dev, generator=gen)
        def c4():
            ti.grad = me.grad = fl.grad = None
            d.softsplat(ti, fl, me, "soft").backward(go)
        ms = _time_cuda(torch, c4, 10, 3)
        px = 8 * 256 * 256
        ex["C4_soft_fwd_bwd_8x64x256x256_f32"] = {"us": round(ms * 1e3, 1), "mpixel_s": round(px / ms / 1e3, 1),
                                                  "alg_gbs": round(1576 * px / ms / 1e6, 1), "frac_of_peak": round(1576 * px / ms / 1e6 / peak, 3)}
        ms = _time_cuda(torch, lambda: d.softsplat(ti.detach(), fl.detach(), me.detach(), "soft"), 10, 3)
        ex["C4_soft_fwd_only_8x64x256x256_f32"] = {"us": round(ms * 1e3, 1), "mpixel_s": round(px / ms / 1e3, 1),
                                                   "alg_gbs": round(131 * 4 * px / ms / 1e6, 1), "frac_of_peak": round(131 * 4 * px / ms / 1e6 / peak, 3)}
        # the same forward on channels_last (NHWC) feature maps: the channel-quad gather (k_list_gather_nhwc); "nchw_gather"
        # is what the same strided view cost before that kernel existed (dcb_set_option("lists_nhwc", 0))
        tcl = ti.detach().to(memory_format=torch.channels_last)
        ms = _time_cuda(torch, lambda: d.softsplat(tcl, fl.detach(), me.detach(), "soft"), 10, 3)
        d._lib.set_option("lists_nhwc", 0)
        ms0 = _time_cuda(torch, lambda: d.softsplat(tcl, fl.detach(), me.detach(), "soft"), 5, 2)
        d._lib.set_option("lists_nhwc", 1)
        ex["C4_soft_fwd_only_channels_last_8x64x256x256_f32"] = {"us": round(ms * 1e3, 1), "mpixel_s": round(px / ms / 1e3, 1),
                                                                 "alg_gbs": round(131 * 4 * px / ms / 1e6, 1),
                                                                 "frac_of_peak": round(131 * 4 * px / ms / 1e6 / peak, 3),
                                                                 "us_through_nchw_gather": round(ms0 * 1e3, 1)}
        del ti, me, fl, go, tcl
        # f-3: Hann-window tile merge (patch_utils.py:83-174): a 1080p canvas from 512^2 tiles with 64 px overlap
        # (patch_exp.ipynb cell 3), at pixel scale (3 channels) and at latent scale (4 channels, 8x smaller)
        def torch_eager_merge(tiles, rects, full):
            # the reference's composition as executed by torch on the same GPU (exact-fit tiles: no resize)
            out = torch.zeros(full, device=dev); weight = torch.zeros_like(out)
            for t, (y1, y2, x1, x2) in zip(tiles, rects):
                wy = torch.hann_window(y2 - y1, periodic=False, device=dev); wx = torch.hann_window(x2 - x1, periodic=False, device=dev)
                m = wy.unsqueeze(1) * wx.unsqueeze(0); m = (m / (m.max() + 1e-12)).expand(1, t.size(1), y2 - y1, x2 - x1)
                out[:, :, y1:y2, x1:x2] += t * m; weight[:, :, y1:y2, x1:x2] += m
            return out / torch.maximum(weight, torch.tensor(1e-8, device=dev))
        for tag, ch, div in (("pixel_3x1080x1920", 3, 1), ("latent_4x135x240", 4, 8)):
            hh, ww, ts, ov = H // div, W // div, 512 // div, 64 // div
            rects = [(y, min(y + ts, hh), x, min(x + ts, ww)) for y in range(0, hh, ts - ov) for x in range(0, ww, ts - ov)]
            tiles = [torch.randn(1, ch, y2 - y1, x2 - x1, device=dev, generator=gen) for (y1, y2, x1, x2) in rects]
            as_read = [(x1, x2, y1, y2) for (y1, y2, x1, x2) in rects]
            ms = _time_cuda(torch, lambda: d.merge_latent_tiles_from_pixel_coords(tiles, as_read, (1, ch, hh, ww), (hh, ww)), 20, 3)
            ms_ref = _time_cuda(torch, lambda: torch_eager_merge(tiles, rects, (1, ch, hh, ww)), 5, 2)
            byts = 4 * (sum(t.numel() for t in tiles) + ch * hh * ww)
            ex[f"f3_tile_merge_{tag}_{len(tiles)}tiles_f32"] = {"us": round(ms * 1e3, 1), "alg_gbs": round(byts / ms / 1e6, 1),
                                                               "frac_of_peak": round(byts / ms / 1e6 / peak, 3),
                                                               "torch_eager_same_gpu_us": round(ms_ref * 1e3, 1)}
    except Exception as e:  # extras must never take the headline line down
        ex["error"] = repr(e)
    return ex


def _reference_gpu(torch, d, dev, gen):
    """B-ref-gpu (BASELINE.md section 5): the reference's OWN, unmodified controlnet/softsplat.py on this GPU -- its eager
    pre/post ops and its three kernel strings, NVRTC-compiled for the device through baseline/cupy_shim.py -- timed next
    to this library on the same tensors: C1 (avg, one 1080p frame), the headline op (soft forward, 16 frames per call)
    and C4 (soft forward + backward, all three gradients, 8 x 64 x 256 x 256)."""
    base = os.path.join(ROOT, "baseline")
    if base not in sys.path:
        sys.path.insert(0, base)
    import ref_gpu
    why = ref_gpu.available()
    if why:
        return {"unavailable": why}
    ref = ref_gpu.load()
    res = {"what": "unmodified reference controlnet/softsplat.py, kernels NVRTC-compiled for this GPU (baseline/cupy_shim.py over cuda-python)"}

    def both(tag, px, mk, iters, warm):
        row = {}
        for name, fn in (("reference", ref.softsplat), ("ours", d.softsplat)):
            ms = _time_cuda(torch, mk(fn), iters, warm)
            row[name + "_us"] = round(ms * 1e3, 1); row[name + "_mpixel_s"] = round(px / ms / 1e3, 1)
        row["speedup"] = round(row["reference_us"] / row["ours_us"], 2)
        res[tag] = row

    t1 = torch.rand(1, 3, H, W, device=dev, generator=gen); f1 = _smooth_flow(torch, 1, H, W, 8.0, dev, gen)
    both("C1_avg_fwd_1x3x1080x1920_f32", H * W, lambda fn: (lambda: fn(tenIn=t1, tenFlow=f1, tenMetric=None, strMode="avg")), 30, 5)
    n = 16
    tn = torch.rand(n, 3, H, W, device=dev, generator=gen); mn = -torch.rand(n, 1, H, W, device=dev, generator=gen)
    fn_ = _smooth_flow(torch, n, H, W, 8.0, dev, gen)
    both("headline_soft_fwd_16x3x1080x1920_f32", n * H * W, lambda fn: (lambda: fn(tenIn=tn, tenFlow=fn_, tenMetric=mn, strMode="soft")), 10, 3)
    # agreement on the headline tensors (atomic order differs: 1e-5 relative is the north star's bound)
    a, b = ref.softsplat(tenIn=tn[:2], tenFlow=fn_[:2], tenMetric=mn[:2], strMode="soft"), d.softsplat(tn[:2], fn_[:2], mn[:2], "soft")
    res["headline_max_abs_diff_over_max_ref"] = float((a - b).abs().max() / a.abs().max())
    del tn, mn, fn_, a, b
    ti = torch.randn(8, 64, 256, 256, device=dev, generator=gen).requires_grad_(True)
    me = (torch.randn(8, 1, 256, 256, device=dev, generator=gen) * 0.5).requires_grad_(True)
    fl = _smooth_flow(torch, 8, 256, 256, 4.0, dev, gen).requires_grad_(True)
    go = torch.randn(8, 64, 256, 256, device=dev, generator=gen)

    def mk4(fn):
        def run():
            ti.grad = me.grad = fl.grad = None
            fn(tenIn=ti, tenFlow=fl, tenMetric=me, strMode="soft").backward(go)
        return run
    both("C4_soft_fwd_bwd_8x64x256x256_f32", 8 * 256 * 256, mk4, 10, 3)
    return res


def _uvg_sweep(torch, d, dev, rank, world, peak, gops_per_chunk=16):
    """C5: the UVG-shaped synthetic 1080p sweep (7 sequences, 3900 frames, 975 GOP-4 units, 2925 inter frames), GOPs
    sharded round-robin over the ranks (STRONG scaling: the sweep is fixed, ranks split it), the conditioning recipe (a-7)
    per inter frame. Every GOP's inputs come from that GOP's own seed, so the per-GOP checksums do not depend on the
    number of ranks. Inputs are generated on the device per chunk (untimed); the recipe is timed with CUDA events; the
    per-GOP checksum table is all-gathered over NCCL afterwards (timed separately)."""
    import torch.distributed as dist
    units = d.shard_units(d.enumerate_gops(), rank, world)
    ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    total_ms, frames, table = 0.0, 0, []
    nmax = gops_per_chunk * 3
    img = torch.empty(nmax, 3, H, W, device=dev); gt = torch.empty(nmax, 3, H, W, device=dev)
    low1 = torch.empty(nmax, 2, H // 32, W // 32, device=dev); low2 = torch.empty_like(low1)
    for i in range(0, len(units), gops_per_chunk):
        chunk = units[i:i + gops_per_chunk]
        n = sum(u.inter_frames for u in chunk)
        at = 0
        for u in chunk:                                               # per-GOP seeds: independent of chunking and sharding
            gen = torch.Generator(device=dev).manual_seed(u.seed())
            k = u.inter_frames
            img[at:at + k].uniform_(generator=gen); gt[at:at + k].uniform_(generator=gen)
            low1[at:at + k].normal_(generator=gen); low2[at:at + k].normal_(generator=gen)
            at += k
        f1 = torch.nn.functional.interpolate(low1[:n], size=(H, W), mode="bicubic", align_corners=False) * 8.0
        f2 = -f1 + 0.5 * torch.nn.functional.interpolate(low2[:n], size=(H, W), mode="bicubic", align_corners=False)
        if i == 0:
            d.residual_conditioning(img[:n], f1, f2, gt[:n], "dataset")          # warm-up, untimed
        torch.cuda.synchronize()
        ev_a.record()
        fused, res = d.residual_conditioning(img[:n], f1, f2, gt[:n], "dataset")
        ev_b.record(); torch.cuda.synchronize()
        total_ms += ev_a.elapsed_time(ev_b); frames += n
        per = res.view(len(chunk), -1)
        table.append(torch.stack([per.sum(dim=1, dtype=torch.float64), (per * per).sum(dim=1, dtype=torch.float64),
                                  torch.full((len(chunk),), float(per.shape[1]), dtype=torch.float64, device=dev)], dim=1))
        del f1, f2, fused, res, per
    local = torch.cat(table) if table else torch.zeros((0, 3), dtype=torch.float64, device=dev)
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    torch.cuda.synchronize()
    g0 = time.perf_counter()
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    allsums = d.gather_checksums(local)                                # [world, kmax, 3] over NCCL (after the sweep, off the timed path)
    torch.cuda.synchronize()
    gather_ms = (time.perf_counter() - g0) * 1e3
    ms = float(t.item())
    all_frames = 2925
    digest = float(allsums[:, :, 0].sum().item())
    # deterministic mode on the first 8 GOPs of the sweep: an exact integer hash of the residual bits, independent of how many
    # ranks shared the work (SURVEY.md App. C-15)
    hashes = torch.zeros(8, dtype=torch.int64, device=dev)
    first_res, first_gi = None, -1
    with d.deterministic(True):
        for gi, u in enumerate(d.enumerate_gops()[:8]):
            if gi % world != rank:
                continue
            gen = torch.Generator(device=dev).manual_seed(u.seed())
            k = u.inter_frames
            img[:k].uniform_(generator=gen); gt[:k].uniform_(generator=gen); low1[:k].normal_(generator=gen); low2[:k].normal_(generator=gen)
            f1 = torch.nn.functional.interpolate(low1[:k], size=(H, W), mode="bicubic", align_corners=False) * 8.0
            f2 = -f1 + 0.5 * torch.nn.functional.interpolate(low2[:k], size=(H, W), mode="bicubic", align_corners=False)
            _, res = d.residual_conditioning(img[:k], f1, f2, gt[:k], "dataset")
            hashes[gi] = res.contiguous().view(torch.int32).to(torch.int64).sum()
            if first_res is None:
                first_res, first_gi = res.clone(), gi
    if world > 1:
        dist.all_reduce(hashes, op=dist.ReduceOp.SUM)                  # exact (integers); every GOP is owned by one rank
    det_hash = int(hashes.sum().item()) & ((1 << 62) - 1)
    # north_star: "NCCL is used only to gather the output tensors": every rank's first deterministic GOP (3 residual frames,
    # 74.6 MB) gathered to rank 0 over NCCL, timed, and checked bit for bit against the hash its owner computed
    out_gather = {"backend": "none"}
    if world > 1 and world <= 8:
        bufs = d.gather_outputs(first_res, dst=0)                     # first use sets up NCCL's point-to-point channels: untimed
        del bufs
        torch.cuda.synchronize(); dist.barrier()
        g1 = time.perf_counter()
        bufs = d.gather_outputs(first_res, dst=0)
        torch.cuda.synchronize()
        og_ms = (time.perf_counter() - g1) * 1e3
        ok = None
        if rank == 0:
            ok = all(int(b.contiguous().view(torch.int32).to(torch.int64).sum().item()) == int(hashes[r].item()) for r, b in enumerate(bufs))
        out_gather = {"backend": "nccl", "tensors": world, "bytes_per_rank": first_res.numel() * first_res.element_size(), "ms": round(og_ms, 2),
                      "gb_s_into_rank0": round((world - 1) * first_res.numel() * first_res.element_size() / og_ms / 1e6, 1),
                      "bit_identical_to_owner_hash": ok}
        del bufs
    return {"gops": 975, "gops_this_rank": len(units), "inter_frames": all_frames, "ms": round(ms, 2), "scaling": "strong",
            "frames_per_s": round(all_frames / ms * 1e3, 1), "mpixel_s": round(all_frames * H * W / ms / 1e3, 1),
            "alg_gbs_per_gpu": round(64 * all_frames * H * W / ms / 1e6 / world, 1),
            "frac_of_peak": round(64 * all_frames * H * W / ms / 1e6 / world / peak, 3),
            "digest": float(f"{digest:.9g}"), "checksum_gather": {"backend": "nccl" if world > 1 else "none", "ms": round(gather_ms, 2),
                                                                   "table": list(allsums.shape)},
            "deterministic_hash_first_8_gops": det_hash, "output_gather": out_gather}


DUMP_SAMPLE = 1 << 22          # elements of the output drawn at fixed positions: 16 MiB in fp32


def _dump_outputs(torch, out, directory):
    """What the last timed step returned, for comparing two builds output for output (the inputs are seeded, so the
    same arguments give the same inputs): frame 0 in full, and the values at DUMP_SAMPLE fixed positions drawn over
    the whole output with a fixed seed, so that every frame of the step is checked. About 42 MB at the bench's sizes."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    flat = out.reshape(-1)
    idx = np.sort(np.random.default_rng(0).integers(0, flat.numel(), size=min(DUMP_SAMPLE, flat.numel())))
    np.save(os.path.join(directory, "softsplat_out_frame0.npy"), out[0].float().cpu().numpy())
    np.save(os.path.join(directory, "softsplat_out_sample.npy"), flat[torch.from_numpy(idx).to(out.device)].float().cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py measures the CUDA path; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    import diffcodec_b200 as d
    numa = d.bind_to_gpu_numa(dev)              # before any pinned allocation: host buffers land next to this GPU's PCIe root

    sampler = ClockSampler(local)               # clocks / throttle reasons from before the warm-up to the end of the timed regions
    if rank == 0:
        sampler.start()

    F = args.frames
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    tin = torch.rand(F, C, H, W, device=dev, generator=gen)
    metric = -torch.rand(F, 1, H, W, device=dev, generator=gen)          # -alpha * photometric error, alpha = 1
    flow = _smooth_flow(torch, F, H, W, 8.0, dev, gen)
    px_per_step = F * H * W

    def step():
        return d.softsplat(tin, flow, metric, "soft")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(max(args.warmup, 3)):
        out = step()
    barrier()
    launches0 = d.launch_count()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    a.record()
    for _ in range(args.steps):
        out = step()
    b.record()
    barrier()
    launches = d.launch_count() - launches0
    ms_step = max_over_ranks(a.elapsed_time(b)) / args.steps
    value = world * px_per_step / ms_step / 1e3                            # Mpixel/s, whole job
    if args.dump_outputs and rank == 0:
        _dump_outputs(torch, out, args.dump_outputs)
    out0 = out[:1].clone()                                                 # for the output check below

    # ---- forward + backward (the other half of BASELINE's metric): all three gradients, 16 frames per GPU per step ----
    nb = min(F, 16)
    ti = tin[:nb].clone().requires_grad_(True); me = metric[:nb].clone().requires_grad_(True); fl = flow[:nb].clone().requires_grad_(True)
    go = torch.randn(nb, C, H, W, device=dev, generator=gen)

    def fb():
        ti.grad = me.grad = fl.grad = None
        d.softsplat(ti, fl, me, "soft").backward(go)
    for _ in range(3):
        fb()
    barrier()
    a.record()
    for _ in range(5):
        fb()
    b.record()
    barrier()
    ms_fb = max_over_ranks(a.elapsed_time(b)) / 5
    del ti, me, fl, go

    # ---- e2e: public API from pinned host buffers, H2D + op + D2H inside the timed region ----
    Fe = min(F, args.e2e_frames)
    h_in = torch.rand(Fe, C, H, W).pin_memory(); h_me = (-torch.rand(Fe, 1, H, W)).pin_memory()
    h_fl = flow[:Fe].cpu().pin_memory(); h_out = torch.empty(Fe, C, H, W).pin_memory()
    # the same frames as a video pipeline holds them: 8-bit pixels, half-precision flow / metric, bf16 result (the latent dtype)
    c_in = (h_in * 255).round().to(torch.uint8).pin_memory(); c_me = h_me.half().pin_memory(); c_fl = h_fl.half().pin_memory()
    c_out = torch.empty(Fe, C, H, W, dtype=torch.bfloat16).pin_memory()

    def time_e2e(fn):
        for _ in range(2):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.e2e_steps):
            fn()
        e1.record()
        barrier()
        return world * Fe * H * W / (max_over_ranks(e0.elapsed_time(e1)) / args.e2e_steps) / 1e3
    e2e_fp32 = time_e2e(lambda: d.softsplat_host(h_in, h_fl, h_me, "soft", out=h_out, device=dev, chunk_frames=8))
    e2e_compact = time_e2e(lambda: d.softsplat_host(c_in, c_fl, c_me, "soft", out=c_out, device=dev, chunk_frames=8))
    # 8-bit / fp16 / bf16 rounding only; a mean, because at hole borders a 0.01 px shift of an fp16 flow flips single pixels between "empty" and "covered"
    e2e_check = float((c_out[:2].float() - h_out[:2]).abs().mean() / h_out[:2].abs().mean())
    del h_in, h_me, h_fl, h_out, c_in, c_me, c_fl, c_out

    # ---- C5: the UVG-shaped sweep sharded by GOP over the ranks (strong scaling) + NCCL gather of the checksums ----
    peak, peak_src = _peaks()
    c5 = None
    if not args.no_c5:
        del tin, metric, flow, out
        torch.cuda.empty_cache()
        try:
            c5 = _uvg_sweep(torch, d, dev, rank, world, peak)
        except Exception as e:
            c5 = {"error": repr(e)}
    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        achieved = ALG_BYTES_PER_PX * px_per_step / ms_step / 1e6          # GB/s per GPU (weak scaling: per-rank time)
        fb_gbs = 112 * nb * H * W / ms_fb / 1e6
        line = {
            "metric": "softsplat soft-mode forward throughput, 1080p fp32 frames", "value": round(value, 1), "unit": "Mpixel/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms_step, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": _config(F),
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                         "traffic": 65.5e6, "traffic_kind": "recorded, not measured in this run",
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of the two launches of one frame (scatter 50.4 + 2.1 MB, normalise 0.2 + 12.8 MB; the rest of the 24.9 MB of output drains after the kernel), ncu --cache-control none, profiles/r02/ncu_step_slots.txt and ncu_step_r02_final.txt; algorithmic 74.65e6",
                         "kernel": "k_splat_step + k_splat_epilogue (two launches per 1080p frame: scatter into one L2-resident accumulator slot, then normalise)",
                         "algorithmic_bytes_per_px": ALG_BYTES_PER_PX, "peak_source": peak_src, "frac_of_nominal_8TBs": round(achieved / 8000.0, 4)},
            "fwd_bwd": {"metric": "softsplat soft-mode forward + backward (gradIn, gradFlow, gradMetric), 1080p fp32 frames",
                        "value": round(world * nb * H * W / ms_fb / 1e3, 1), "unit": "Mpixel/s", "ms_per_step": round(ms_fb, 3), "frames_per_gpu": nb,
                        "algorithmic_bytes_per_px": 112, "achieved_gbs_per_gpu": round(fb_gbs, 1), "frac": round(fb_gbs / peak, 4)},
            "e2e": {"value": round(e2e_compact, 1), "unit": "Mpixel/s", "h2d_bytes_per_step": Fe * (C + 2 * 3) * H * W,
                    "d2h_bytes_per_step": Fe * C * H * W * 2, "frames_per_step": Fe,
                    "api": "diffcodec_b200.softsplat_host(frames uint8, flow fp16, metric fp16, 'soft', out=pinned bf16): pinned host tensors in and out, "
                           "copies and the on-device widening to fp32 inside the timed region, synchronous return",
                    "element_types": "uint8 frames (decoded video), fp16 flow and metric, bf16 result (the latent dtype); the splat runs in fp32",
                    "mean_abs_diff_vs_fp32_path_over_mean_abs": round(e2e_check, 5),
                    "fp32_host_tensors": {"value": round(e2e_fp32, 1), "unit": "Mpixel/s", "h2d_bytes_per_step": Fe * (C + 3) * H * W * 4,
                                          "d2h_bytes_per_step": Fe * C * H * W * 4}},
            "gpu_launches": int(launches), "clocks": clocks, "numa": numa,
            "c5_uvg_sweep": c5,
        }
        if world == 1 and not args.no_cpu:
            from oracle import oracle as orc
            threads = orc.max_threads()
            nsample = max(4, (F // max(threads, 1)) * threads) if F >= threads else F      # whole rounds of the thread pool
            v, secs = _cpu_port_mpixel_s(nsample, threads, repeats=2)
            line["cpu_baseline"] = {"value": round(v, 2), "unit": "Mpixel/s", "cores": threads, "kind": "port",
                                    "sample": f"{nsample} of the step's {F} 1080p frames, soft fwd fp32, best of 2 runs of {secs:.1f} s = "
                                              f"{secs * threads:.0f} core-seconds (oracle C kernel over {threads} pthreads + torch CPU pre/post ops)"}
            # the oracle as CHECKER of what was timed: frame 0 of the timed step's inputs, CPU port vs the GPU result
            try:
                g0 = torch.Generator(device=dev).manual_seed(1234 + rank)
                t0 = torch.rand(F, C, H, W, device=dev, generator=g0)[:1].cpu(); m0 = (-torch.rand(F, 1, H, W, device=dev, generator=g0))[:1].cpu()
                f0 = _smooth_flow(torch, F, H, W, 8.0, dev, g0)[:1].cpu()
                ref0 = orc.softsplat(t0, f0, m0, "soft")
                line["output_check"] = {"what": "frame 0 of the timed step vs the CPU oracle", "max_abs_diff_over_max": float((out0.cpu() - ref0).abs().max() / ref0.abs().max()),
                                        "tolerance": 1e-5}
            except Exception as e:
                line["output_check"] = {"error": repr(e)}
        else:
            line["cpu_baseline"] = None
        if world == 1 and not args.no_extra:
            torch.cuda.empty_cache()
            line["extra"] = _extras(torch, d, dev, gen, peak)
            try:
                line["extra"]["reference_gpu"] = _reference_gpu(torch, d, dev, gen)
            except Exception as e:
                line["extra"]["reference_gpu"] = {"error": repr(e)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=64, help="1080p frames per GPU per step")
    ap.add_argument("--e2e-frames", type=int, default=64)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="skip the UVG-shaped sweep (C5)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed sample of the last step's output (rank 0) as DIR/*.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
