"""fp16 against bf16 (and fp32) on the conditioning path, CUDA events after warm-up, every variant alternated over several
rounds in one process (median and min..max spread of the rounds):

  * the live consumer's four-scale pyramid (Bi_Dir_FeatureExtractor, batch 2) forward + backward, eager and as one CUDA-graph
    replay: fp32, bf16, native fp16, and fp16 computed by casting every input to fp32 and every output / gradient back (the
    composition native fp16 replaces), with the library launches and all CUDA kernels of one step;
  * softsplat(..., "soft") forward on the bench's 64 x 3 x 1080 x 1920 frames, fp16 and bf16;
  * the C4 shape 8 x 64 x 256 x 256 forward + backward (per-target lists), NCHW and channels_last, fp16 and bf16;
  * the 15-tile merge of a 1080p frame (512-pixel tiles), fp16 and bf16.

    python profiles/scripts/fp16_paths.py --out OUT.json [--rounds 5]

Needs a GPU; the card's name and power limit are read in the same run and written next to the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import diffcodec_b200 as d  # noqa: E402

LIVE = [(2, 160, 64, 64), (2, 160, 32, 32), (2, 320, 16, 16), (2, 640, 8, 8)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def time_eager(fn, iters):
    for _ in range(3):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e3


def make_graph(fn):
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
    return graph.replay


def kernels_of(fn):
    """CUDA kernels of one call, from the profiler (a run of its own, not a timed one)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "Memset" not in e.name and "Memcpy" not in e.name)


def pyramid_step(dtype, cast=False):
    g = torch.Generator().manual_seed(1)
    store = torch.float16 if cast else dtype
    levels = []
    for n, c, h, w in LIVE:
        ff = torch.randn(n, 2, h, w, generator=g) * 0.6
        vals = (torch.randn(n, c, h, w, generator=g), torch.randn(n, c, h, w, generator=g), ff, -ff + 0.25 * torch.randn(n, 2, h, w, generator=g),
                torch.randn(n, 1, h, w, generator=g) * 0.5 + 0.1, torch.randn(n, 1, h, w, generator=g) * 0.5 + 0.1)
        levels.append([v.to(store).cuda().requires_grad_(True) for v in vals])
    gouts = [torch.randn(lv[0].shape, generator=g).to(store).cuda() for lv in levels]
    leaves = [t for lv in levels for t in lv]

    def step():
        for t in leaves:
            t.grad = None
        if cast:       # the composition: every input to fp32, the fp32 library call, every output back (autograd casts the gradients)
            outs = [o.half() for o in d.bidirectional_pyramid([tuple(t.float() for t in lv) for lv in levels])]
        else:
            outs = d.bidirectional_pyramid([tuple(lv) for lv in levels])
        torch.autograd.backward(outs, gouts)
    return step


def splat_1080p(dtype):
    g = torch.Generator(device="cuda").manual_seed(2)
    x = torch.randn(64, 3, 1080, 1920, generator=g, device="cuda").to(dtype)
    fl = (torch.randn(64, 2, 1080, 1920, generator=g, device="cuda") * 2).to(dtype)
    m = (torch.randn(64, 1, 1080, 1920, generator=g, device="cuda") * 0.5).to(dtype)
    return lambda: d.softsplat(x, fl, m, "soft")


def c4_step(dtype, channels_last):
    g = torch.Generator().manual_seed(3)
    x = torch.randn(8, 64, 256, 256, generator=g).to(dtype).cuda()
    if channels_last:
        x = x.to(memory_format=torch.channels_last)
    x.requires_grad_(True)
    fl = (torch.randn(8, 2, 256, 256, generator=g) * 2).to(dtype).cuda().requires_grad_(True)
    m = (torch.randn(8, 1, 256, 256, generator=g) * 0.5).to(dtype).cuda().requires_grad_(True)
    gout = torch.randn(8, 64, 256, 256, generator=g).to(dtype).cuda()

    def step():
        for t in (x, fl, m):
            t.grad = None
        d.softsplat(x, fl, m, "soft").backward(gout)
    return step


def merge_1080p(dtype):
    xs, ys = (0, 352, 704, 1056, 1408), (0, 284, 568)
    coords = [(x, x + 512, y, y + 512) for y in ys for x in xs]
    g = torch.Generator().manual_seed(4)
    lat = [torch.randn(1, 4, 64, 64, generator=g).to(dtype).cuda() for _ in coords]
    return lambda: d.merge_latent_tiles_from_pixel_coords(lat, coords, (1, 4, 135, 240), (1080, 1920))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "fp16_paths.py measures on the GPU"
    torch.backends.cudnn.allow_tf32 = False
    H, B, F32 = torch.float16, torch.bfloat16, torch.float32
    cases = {}          # name -> (fn, iters)
    for name, dt, cast in (("fp32", F32, False), ("bf16", B, False), ("fp16", H, False), ("fp16_via_fp32_casts", H, True)):
        cases[f"pyramid_live_b2_fwd_bwd_{name}_eager_us"] = (pyramid_step(dt, cast), 200)
    for name, dt in (("fp16", H), ("bf16", B)):
        cases[f"softsplat_soft_64x3x1080x1920_{name}_us"] = (splat_1080p(dt), 10)
        cases[f"c4_8x64x256x256_fwd_bwd_nchw_{name}_us"] = (c4_step(dt, False), 20)
        cases[f"c4_8x64x256x256_fwd_bwd_channels_last_{name}_us"] = (c4_step(dt, True), 20)
        cases[f"tile_merge_15x1080p_{name}_us"] = (merge_1080p(dt), 500)
    res = {"card": card(), "rounds": args.rounds, "launches": {}}
    for key, (fn, _) in cases.items():
        if key.startswith("pyramid"):
            fn()
            before = d.launch_count()
            fn()
            torch.cuda.synchronize()
            res["launches"][key.replace("_eager_us", "")] = {"library": d.launch_count() - before, "cuda_kernels": kernels_of(fn)}
    graphs = {k.replace("_eager_us", "_graph_us"): make_graph(fn) for k, (fn, _) in cases.items() if k.startswith("pyramid")}
    samples = {k: [] for k in list(cases) + list(graphs)}
    for _ in range(args.rounds):                 # variants alternate inside every round
        for key, (fn, iters) in cases.items():
            samples[key].append(time_eager(fn, iters))
        for key, replay in graphs.items():
            samples[key].append(time_eager(replay, 500))
    res["times_us"] = {k: {"median": statistics.median(v), "min": min(v), "max": max(v)} for k, v in samples.items()}
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
