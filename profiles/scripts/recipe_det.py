"""The conditioning recipes under deterministic() in two arms, fp32:

  det_call      residual_conditioning / residual_conditioning_bidir as they run now: one dcb_residual_fused / dcb_residual_bidir
                call with DCB_FLAG_DETERMINISTIC per frame group (emit, one radix sort, reduce, fuse: 11 launches)
  det_composed  what they ran before (residual_utils._composed / _composed_bidir): three (bidir: four) deterministic soft
                splats, each emit + sort + reduce + normalise, and the torch ops of the mask norms, the fusion and the residual

    python profiles/scripts/recipe_det.py --out profiles/r07

Workloads:
  c5_hash     the deterministic hash of bench.py's C5 record: 8 GOPs x 3 inter frames at 1080p, one call per GOP, the same
              per-GOP seeded inputs; the hash of the residual bits is recorded for both arms
  64x1080p    one call on 64 frames of 1080p (the library path splits it into frame groups)
  512         the reference's per-sample call, [1,3,512,512]

Eager (CUDA events around `iters` calls) and as a CUDA-graph replay; the arms alternate inside each round and the JSON keeps
the median over rounds. Launches: the library's own launch counter for one call, and the CUDA kernels and memsets of one call
as torch.profiler lists them (the composition's torch ops included). The card's name, power limit and clock limit are read in
the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))   # the repository root

H, W = 1080, 1920


def c5_inputs(torch, d, dev):
    """bench.py's deterministic-hash inputs: per GOP (img, f1, f2, gt) from the GOP's own seed."""
    F = torch.nn.functional
    out = []
    for u in d.enumerate_gops()[:8]:
        gen = torch.Generator(device=dev).manual_seed(u.seed())
        k = u.inter_frames
        img, gt = torch.empty(k, 3, H, W, device=dev), torch.empty(k, 3, H, W, device=dev)
        low1, low2 = torch.empty(k, 2, H // 32, W // 32, device=dev), torch.empty(k, 2, H // 32, W // 32, device=dev)
        img.uniform_(generator=gen); gt.uniform_(generator=gen); low1.normal_(generator=gen); low2.normal_(generator=gen)
        f1 = F.interpolate(low1, size=(H, W), mode="bicubic", align_corners=False) * 8.0
        f2 = -f1 + 0.5 * F.interpolate(low2, size=(H, W), mode="bicubic", align_corners=False)
        out.append((img, f1, f2, gt))
    return out


def frames(torch, n, h, w, seed, dev):
    F = torch.nn.functional
    g = torch.Generator(device=dev).manual_seed(seed)
    img1, img2, gt = (torch.rand(n, 3, h, w, device=dev, generator=g) for _ in range(3))
    low = torch.randn(n, 2, h // 32, w // 32, device=dev, generator=g)
    f1 = F.interpolate(low, size=(h, w), mode="bicubic", align_corners=False) * 8.0
    f2 = -f1 + 0.5 * torch.randn(n, 2, h, w, device=dev, generator=g)
    return img1, img2, f1, f2, gt


def timed(torch, fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e3


def capture(torch, fn):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        fn()
    torch.cuda.synchronize()
    return graph


def device_ops(torch, fn):
    """CUDA kernels + memsets of one call, as torch.profiler lists them."""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r07")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=5)
    a = ap.parse_args()
    import importlib
    import torch
    import diffcodec_b200 as d
    ru = importlib.import_module(d.__name__ + ".residual_utils")
    assert torch.cuda.is_available(), "this script measures on the GPU"
    dev = torch.device("cuda")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": gpu, "rounds": a.rounds, "iters": a.iters, "det_group_bytes": ru.DET_GROUP_BYTES, "launches": {},
           "device_ops": {}, "graph_errors": {}, "equal": {}, "samples": {}}

    c5 = c5_inputs(torch, d, dev)
    big = frames(torch, 64, H, W, 5, dev)
    small = frames(torch, 1, 512, 512, 6, dev)
    res["frames_per_group"] = {"c5_hash": ru._det_group(3, 3, H, W)[0], "64x1080p": ru._det_group(64, 3, H, W)[0],
                               "512": ru._det_group(1, 3, 512, 512)[0]}

    def call(kind, img1, img2, f1, f2, gt):
        if kind == "bidir":
            return d.residual_conditioning_bidir(img1, img2, f1, f2, gt, return_masks=True)
        return d.residual_conditioning(img1, f1, f2, gt, kind, return_masks=True)

    def composed(kind, img1, img2, f1, f2, gt):
        if kind == "bidir":
            return ru._composed_bidir(img1, img2, f1, f2, gt)
        return ru._composed(img1, f1, f2, gt, kind)

    arms = {"det_call": call, "det_composed": composed}
    steps = {}
    for arm, fn in arms.items():
        def c5_step(fn=fn):
            with torch.no_grad(), d.deterministic():
                return [fn("dataset", img, None, f1, f2, gt) for img, f1, f2, gt in c5]
        steps[f"c5_hash_dataset_{arm}"] = c5_step
        for kind in ("dataset", "bidir"):
            for name, ins in (("64x1080p", big), ("512", small)):
                def step(fn=fn, kind=kind, ins=ins):
                    with torch.no_grad(), d.deterministic():
                        return fn(kind, *ins)
                steps[f"{name}_{kind}_{arm}"] = step

    # bit equality of the two arms on every workload, and the C5 hash of both
    for key, step in steps.items():
        if not key.endswith("_det_call"):
            continue
        base = key[:-len("_det_call")]
        got, ref = step(), steps[base + "_det_composed"]()
        if base.startswith("c5"):
            res["c5_hash"] = {}
            for arm, outs in (("det_call", got), ("det_composed", ref)):
                h = sum(int(o[1].contiguous().view(torch.int32).to(torch.int64).sum()) for o in outs) & ((1 << 62) - 1)
                res["c5_hash"][arm] = h
            got, ref = [t for o in got for t in o], [t for o in ref for t in o]
        res["equal"][base] = all(bool(torch.equal(x, y)) for x, y in zip(got, ref))
        del got, ref
    for key, step in steps.items():
        step()
        before = d.launch_count()
        step()
        torch.cuda.synchronize()
        res["launches"][key] = d.launch_count() - before
        try:
            res["device_ops"][key] = device_ops(torch, step)
        except Exception as e:                                     # reported, not hidden
            res["device_ops"][key] = f"error: {str(e).splitlines()[0][:200]}"
    timed_steps = {k + "_eager_us": v for k, v in steps.items()}
    keep = []                                                      # every workspace a captured graph points at stays alive
    for key, step in steps.items():
        try:
            timed_steps[key + "_graph_us"] = capture(torch, step).replay
            keep.extend(d._lib._workspaces.values())
        except Exception as e:                                     # reported, not hidden: the eager numbers stand
            torch.cuda.synchronize()
            res["graph_errors"][key] = str(e).splitlines()[0][:200]
    for fn in timed_steps.values():                                # warm every timed path once more
        fn()
    for r in range(a.rounds):
        for key, fn in timed_steps.items():                        # arms alternate inside each round
            res["samples"].setdefault(key, []).append(timed(torch, fn, a.iters))
    res["median_us"] = {k: sorted(v)[len(v) // 2] for k, v in res["samples"].items()}
    res["when"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "recipe_det_b200.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "samples"}, indent=1))


if __name__ == "__main__":
    main()
