"""The motion compensation of Bi_Dir_FeatureExtractor (four scales, batch 2: (160, 64), (160, 32), (320, 16), (640, 8)) in three
arms, fp32 and bf16:

  plain        bidirectional_pyramid (dcb_bidir_pyramid_fwd / _bwd: two launches each way)
  det_pyramid  the same call under deterministic() (emit, one radix sort, reduce, fuse)
  det_composed what the extractor ran under deterministic() before the pyramid honoured the flag: per scale compute_mask x2,
               two masked deterministic soft splats, bidir_fuse

    python profiles/scripts/pyramid_det.py --out profiles/r06

Forward alone (inference: no input requires a gradient) and forward + backward (features, metrics and flows require one),
eager and as a CUDA-graph replay; CUDA events around `iters` calls; the arms alternate inside each round and the JSON keeps
the median over rounds. The card's name, power limit and clock limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))   # the repository root

SHAPES = [(2, 160, 64), (2, 160, 32), (2, 320, 16), (2, 640, 8)]


def inputs(torch, dtype):
    g = torch.Generator().manual_seed(7)
    levels, gouts = [], []
    for n, c, r in SHAPES:
        first, last = torch.randn(n, c, r, r, generator=g), torch.randn(n, c, r, r, generator=g)
        ff = torch.randn(n, 2, r, r, generator=g) * 0.6
        fb = -ff + 0.25 * torch.randn(n, 2, r, r, generator=g)
        mf, mb = torch.randn(n, 1, r, r, generator=g) * 0.5 + 0.1, torch.randn(n, 1, r, r, generator=g) * 0.5 + 0.1
        levels.append([t.cuda().to(dtype) for t in (first, last, ff, fb, mf, mb)])
        gouts.append(torch.randn(n, c, r, r, generator=g).cuda().to(dtype))
    return levels, gouts


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r06")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=50)
    a = ap.parse_args()
    import torch
    import diffcodec_b200 as d
    import importlib
    ss = importlib.import_module(d.__name__ + ".softsplat")
    assert torch.cuda.is_available(), "this script measures on the GPU"
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()

    def composed(levels):
        outs = []
        for first, last, ff, fb, mf, mb in levels:
            of, ob = d.compute_mask(ff, fb), d.compute_mask(fb, ff)
            wa = ss._splat_normalised(first, ff, mf, d._lib.MODE_SOFT, d._lib.EPS_ADD, mask=of)
            wb = ss._splat_normalised(last, fb, mb, d._lib.MODE_SOFT, d._lib.EPS_ADD, mask=ob)
            outs.append(d.bidir_fuse(wa, wb, mf, mb, of, ob))
        return outs

    arms = {"plain": (False, lambda lv: d.bidirectional_pyramid([tuple(x) for x in lv])),
            "det_pyramid": (True, lambda lv: d.bidirectional_pyramid([tuple(x) for x in lv])),
            "det_composed": (True, composed)}
    res = {"gpu": gpu, "shapes": SHAPES, "rounds": a.rounds, "iters": a.iters, "launches": {}, "graph_errors": {}, "samples": {}}
    steps = {}
    for dtype in (torch.float32, torch.bfloat16):
        dn = str(dtype).split(".")[-1]
        levels, gouts = inputs(torch, dtype)
        grad_levels = [[t.clone().requires_grad_(True) for t in lv] for lv in levels]
        leaves = [t for lv in grad_levels for t in lv]
        for arm, (det, fn) in arms.items():
            def fwd(det=det, fn=fn):
                with torch.no_grad(), d.deterministic(det):
                    return fn(levels)

            def fwd_bwd(det=det, fn=fn):
                for t in leaves:
                    t.grad = None
                with d.deterministic(det):
                    outs = fn(grad_levels)
                torch.autograd.backward(outs, gouts)

            for mode, step in (("fwd", fwd), ("fwd_bwd", fwd_bwd)):
                key = f"{dn}_{mode}_{arm}"
                step()
                before = d.launch_count()
                step()
                torch.cuda.synchronize()
                res["launches"][key] = d.launch_count() - before
                steps[key + "_eager_us"] = step
    graphs = {}
    for key, step in list(steps.items()):                          # captures last: a failed one ends the captures
        try:
            graphs[key.replace("_eager_us", "_graph_us")] = capture(torch, step).replay
        except Exception as e:                                     # reported, not hidden: the eager numbers stand
            torch.cuda.synchronize()
            res["graph_errors"][key] = str(e).splitlines()[0][:200]
            break
    steps.update(graphs)
    # the outputs the timed calls produce: deterministic pyramid vs deterministic composition (fp32: bit-identical expected)
    for dtype in (torch.float32, torch.bfloat16):
        dn = str(dtype).split(".")[-1]
        levels, _ = inputs(torch, dtype)
        with torch.no_grad(), d.deterministic():
            p, c = d.bidirectional_pyramid([tuple(x) for x in levels]), composed(levels)
        res[f"{dn}_det_pyramid_equals_composition"] = all(bool(torch.equal(x, y)) for x, y in zip(p, c))
        res[f"{dn}_det_pyramid_vs_composition_max_abs"] = max(float((x.float() - y.float()).abs().max()) for x, y in zip(p, c))
    for fn in steps.values():                                      # warm every timed path once more
        for _ in range(5):
            fn()
    for r in range(a.rounds):
        for key, fn in steps.items():                              # arms alternate inside each round
            res["samples"].setdefault(key, []).append(timed(torch, fn, a.iters))
    res["median_us"] = {k: sorted(v)[len(v) // 2] for k, v in res["samples"].items()}
    res["when"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "pyramid_det_live_batch2.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "samples"}, indent=1))


if __name__ == "__main__":
    main()
