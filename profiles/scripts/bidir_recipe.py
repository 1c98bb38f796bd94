#!/usr/bin/env python
"""Two-reference conditioning builder (dcb_residual_bidir) on a B200, in one run:

  1. 64 x 3 x 1080 x 1920 in fp32 and bf16 (inputs ~4.5 GB in fp32, far above the 126 MB L2): the fused entry
     (residual_conditioning_bidir), the composition of single-op calls it replaces (softsplat x2, compute_mask x2, bidir_fuse,
     subtraction) and the one-reference recipe (residual_conditioning), interleaved per repetition, CUDA events, median of
     --reps. Gpx/s and GB/s on algorithmic bytes, (5C+4)*s per pixel for the two-reference recipe (read both images, both flows
     and gt; write fused and residual) and (3C+4)*s for the one-reference recipe, as a fraction of bench.py's HBM figure.
     Kernel launches per call (library count; all CUDA kernels from torch.profiler) and the max |fused - composed| away
     from mask flips.
  2. The UVG-shaped sweep of C5 (975 GOPs of 4, 2925 inter frames, per-GOP seeds as bench.py _uvg_sweep; each GOP brings
     two I-frames, repeated over its three inter frames outside the timed region) through the two-reference builder, and
     the one-reference recipe on the same inputs, both timed per chunk with CUDA events.

    python profiles/scripts/bidir_recipe.py --out profiles/r03/bidir_recipe_64x1080p_and_uvg_sweep.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

H, W, C = 1080, 1920, 3


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_clock_max"] = (x.strip() for x in out.split(","))
    except Exception as e:  # the numbers stay meaningful with the card name; say why the rest is missing
        info["nvidia_smi"] = repr(e)
    return info


def kernels_per_call(torch, fn):
    """CUDA kernels of one call, from torch.profiler (library kernels and torch's own)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in p.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kern = [n for n in names if not n.startswith(("Memset", "Memcpy", "[Memset", "[Memcpy"))]
    return {"kernels": len(kern), "memsets": len(names) - len(kern)}


def timed_64(torch, d, ru, dtype, reps, peak):
    n = 64
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(7)
    import bench
    img1 = torch.rand(n, C, H, W, device=dev, generator=gen).to(dtype)
    img2 = torch.rand(n, C, H, W, device=dev, generator=gen).to(dtype)
    gt = torch.rand(n, C, H, W, device=dev, generator=gen).to(dtype)
    f1 = bench._smooth_flow(torch, n, H, W, 8.0, dev, gen)
    f2 = (-f1 + 0.5 * bench._smooth_flow(torch, n, H, W, 1.0, dev, gen)).to(dtype)
    f1 = f1.to(dtype)
    calls = {
        "fused_bidir": lambda: d.residual_conditioning_bidir(img1, img2, f1, f2, gt),
        "composed_bidir": lambda: ru._composed_bidir(img1, img2, f1, f2, gt),
        "one_reference_recipe": lambda: d.residual_conditioning(img1, f1, f2, gt, "dataset"),
    }
    with torch.no_grad():
        for fn in calls.values():
            for _ in range(2):
                fn()
        torch.cuda.synchronize()
        times = {k: [] for k in calls}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for _ in range(reps):                         # alternate the three in every repetition
            for k, fn in calls.items():
                ev[0].record()
                fn()
                ev[1].record()
                torch.cuda.synchronize()
                times[k].append(ev[0].elapsed_time(ev[1]))
        s = torch.finfo(dtype).bits // 8
        res = {}
        for k, fn in calls.items():
            ms = statistics.median(times[k])
            bpp = (5 * C + 4) * s if k != "one_reference_recipe" else (3 * C + 4) * s
            l0 = d.launch_count(); fn(); torch.cuda.synchronize()
            row = {"ms_median": round(ms, 3), "ms_min": round(min(times[k]), 3), "ms_max": round(max(times[k]), 3),
                   "gpx_s": round(n * H * W / ms / 1e6, 2), "alg_bytes_per_px": bpp, "alg_gbs": round(bpp * n * H * W / ms / 1e6, 1),
                   "frac_of_hbm_peak": round(bpp * n * H * W / ms / 1e6 / peak, 3), "library_launches_per_call": d.launch_count() - l0}
            try:
                row["cuda_kernels_per_call"] = kernels_per_call(torch, fn)
            except Exception as e:
                row["cuda_kernels_per_call"] = repr(e)
            res[k] = row
        fused, resid, of, ob = d.residual_conditioning_bidir(img1, img2, f1, f2, gt, return_masks=True)
        fc, rc, ofc, obc = ru._composed_bidir(img1, img2, f1, f2, gt)
        same = ((of == ofc) & (ob == obc)).expand_as(fused)
        res["fused_vs_composed"] = {
            "mask_pixels_differing": int((~((of == ofc) & (ob == obc))).sum()), "pixels": n * H * W,
            "max_abs_diff_fused_where_masks_agree": float((fused.float() - fc.float()).abs()[same].max()),
            "max_abs_diff_residual_where_masks_agree": float((resid.float() - rc.float()).abs()[same].max()),
            "occ_fwd_mean": float(of.float().mean()), "occ_bwd_mean": float(ob.float().mean())}
        res["speedup_fused_over_composed"] = round(res["composed_bidir"]["ms_median"] / res["fused_bidir"]["ms_median"], 2)
        res["reps"] = reps
    del img1, img2, gt, f1, f2, fused, resid, of, ob, fc, rc, ofc, obc, same
    torch.cuda.empty_cache()
    return res


def uvg_sweep(torch, d, gops_per_chunk=16):
    dev = torch.device("cuda", 0)
    units = d.enumerate_gops()
    nmax = gops_per_chunk * 3
    i1 = torch.empty(gops_per_chunk, C, H, W, device=dev); i2 = torch.empty_like(i1)
    gt = torch.empty(nmax, C, H, W, device=dev)
    low1 = torch.empty(nmax, 2, H // 32, W // 32, device=dev); low2 = torch.empty_like(low1)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    ms_bidir = ms_one = 0.0
    frames, dig_bidir, dig_one = 0, 0.0, 0.0
    with torch.no_grad():
        for i in range(0, len(units), gops_per_chunk):
            chunk = units[i:i + gops_per_chunk]
            n, at, rep = sum(u.inter_frames for u in chunk), 0, []
            for j, u in enumerate(chunk):                                 # per-GOP seeds: independent of chunking
                gen = torch.Generator(device=dev).manual_seed(u.seed())
                k = u.inter_frames
                i1[j].uniform_(generator=gen); i2[j].uniform_(generator=gen)
                gt[at:at + k].uniform_(generator=gen)
                low1[at:at + k].normal_(generator=gen); low2[at:at + k].normal_(generator=gen)
                rep += [j] * k
                at += k
            idx = torch.tensor(rep, device=dev)
            img1, img2 = i1.index_select(0, idx), i2.index_select(0, idx)   # each I-frame pair over its GOP's inter frames
            f1 = torch.nn.functional.interpolate(low1[:n], size=(H, W), mode="bicubic", align_corners=False) * 8.0
            f2 = -f1 + 0.5 * torch.nn.functional.interpolate(low2[:n], size=(H, W), mode="bicubic", align_corners=False)
            if i == 0:                                                    # warm-up, untimed
                d.residual_conditioning_bidir(img1, img2, f1, f2, gt[:n]); d.residual_conditioning(img1, f1, f2, gt[:n], "dataset")
            torch.cuda.synchronize()
            ev[0].record()
            _, rb = d.residual_conditioning_bidir(img1, img2, f1, f2, gt[:n])
            ev[1].record()
            ev[2].record()
            _, ro = d.residual_conditioning(img1, f1, f2, gt[:n], "dataset")
            ev[3].record()
            torch.cuda.synchronize()
            ms_bidir += ev[0].elapsed_time(ev[1]); ms_one += ev[2].elapsed_time(ev[3])
            dig_bidir += float(rb.sum(dtype=torch.float64)); dig_one += float(ro.sum(dtype=torch.float64))
            frames += n
            del img1, img2, f1, f2, rb, ro
    return {"gops": len(units), "inter_frames": frames, "i_frames_per_gop": 2, "dtype": "float32",
            "two_reference_ms": round(ms_bidir, 2), "one_reference_ms": round(ms_one, 2),
            "two_reference_frames_per_s": round(frames / ms_bidir * 1e3, 1), "one_reference_frames_per_s": round(frames / ms_one * 1e3, 1),
            "two_reference_over_one_reference": round(ms_bidir / ms_one, 3),
            "residual_digest_two_reference": float(f"{dig_bidir:.9g}"), "residual_digest_one_reference": float(f"{dig_one:.9g}")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    ap.add_argument("--reps", type=int, default=21)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bidir_recipe.py measures on the GPU; none is visible")
    import diffcodec_b200 as d
    import bench
    from importlib import import_module
    ru = import_module(d.__name__ + ".residual_utils")
    peak, peak_src = bench._peaks()
    out = {"card": card(), "hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "torch": torch.__version__,
           "shape": [64, C, H, W], "l2_policy": "inputs of one call 4.5 GB (fp32) / 2.2 GB (bf16), far above the 126 MB L2"}
    for name, dt in (("float32", torch.float32), ("bfloat16", torch.bfloat16)):
        out[f"batch64_{name}"] = timed_64(torch, d, ru, dt, args.reps, peak)
    out["uvg_sweep_c5_shape"] = uvg_sweep(torch, d)
    out["card_after"] = card()
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
