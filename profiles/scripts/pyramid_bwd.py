"""Forward + backward of the conditioning pyramid's motion compensation at the live consumer's sizes (four scales, batch 2:
(160, 64), (160, 32), (320, 16), (640, 8)), old and new side by side in one run.

    python profiles/scripts/pyramid_bwd.py --parent build_variants/parent --out profiles/r04

--parent is a built checkout of the parent commit (git archive + make). Each round runs one worker process per tree,
alternating. A worker times, with CUDA events:
  * bidirectional_pyramid + its backward (features and metrics require a gradient, flows do not: what both trees support),
    fp32 and bf16, eager and as one CUDA-graph replay;
  * in the new tree only: the motion compensation of Bi_Dir_ResidueExtractor (flows require a gradient) as the composition
    the parent ran (compute_mask x2, two masked splats, bidir_fuse, per scale) and as one bidirectional_pyramid(holes=False),
    with the launches of one forward + backward.
Before timing, both trees store their outputs and gradients at the timed sizes; the parent compares them afterwards.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

SHAPES = [(2, 160, 64), (2, 160, 32), (2, 320, 16), (2, 640, 8)]


def inputs(torch, dtype, flow_grad=False):
    g = torch.Generator().manual_seed(7)
    levels, gouts = [], []
    for n, c, r in SHAPES:
        first, last = torch.randn(n, c, r, r, generator=g), torch.randn(n, c, r, r, generator=g)
        ff = torch.randn(n, 2, r, r, generator=g) * 0.6
        fb = -ff + 0.25 * torch.randn(n, 2, r, r, generator=g)
        mf, mb = torch.randn(n, 1, r, r, generator=g) * 0.5 + 0.1, torch.randn(n, 1, r, r, generator=g) * 0.5 + 0.1
        lv = [t.cuda().to(dtype) for t in (first, last, ff, fb, mf, mb)]
        for k in (0, 1, 4, 5) + ((2, 3) if flow_grad else ()):
            lv[k].requires_grad_(True)
        levels.append(lv)
        gouts.append(torch.randn(n, c, r, r, generator=g).cuda().to(dtype))
    return levels, gouts


def time_eager(torch, fn, iters=200, warm=20):
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e3


def time_graph(torch, fn, iters=500):
    try:
        return _time_graph(torch, fn, iters)
    except Exception as e:                                          # reported, not hidden: the eager numbers stand
        torch.cuda.synchronize()
        return "capture failed: " + str(e).splitlines()[0]


def _time_graph(torch, fn, iters):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(5):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        fn()
    for _ in range(20):
        graph.replay()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        graph.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e3


def worker(tree, out_dir, label):
    sys.path.insert(0, tree)
    import torch
    import diffcodec_b200 as d
    res = {"tree": label}
    dump, graphs = {}, []                                           # graph captures last: a failed one ends the worker's timings
    for dtype in (torch.float32, torch.bfloat16):
        name = str(dtype).split(".")[-1]
        levels, gouts = inputs(torch, dtype)
        leaves = [t for lv in levels for t in lv if t.requires_grad]

        def step():
            for t in leaves:
                t.grad = None
            outs = d.bidirectional_pyramid([tuple(lv) for lv in levels])
            torch.autograd.backward(outs, gouts)
            return outs

        outs = step()
        dump[name] = [o.detach().float().cpu() for o in outs] + [t.grad.float().cpu() for t in leaves]
        before = d.launch_count()
        step()
        torch.cuda.synchronize()
        res[f"{name}_launches_fwd_bwd"] = d.launch_count() - before
        res[f"{name}_eager_us"] = time_eager(torch, step)
        graphs.append((f"{name}_graph_us", step))
    torch.save(dump, os.path.join(out_dir, f"parity_{label}.pt"))           # a temporary directory (main)
    if label == "this":
        import importlib
        ss = importlib.import_module(d.__name__ + ".softsplat")
        levels, gouts = inputs(torch, torch.float32, flow_grad=True)
        leaves = [t for lv in levels for t in lv if t.requires_grad]

        def composed():
            outs = []
            for first, last, ff, fb, mf, mb in levels:
                of, ob = d.compute_mask(ff, fb), d.compute_mask(fb, ff)
                wa = ss._splat_normalised(first, ff, mf, d._lib.MODE_SOFT, d._lib.EPS_ADD, mask=of)
                wb = ss._splat_normalised(last, fb, mb, d._lib.MODE_SOFT, d._lib.EPS_ADD, mask=ob)
                outs.append(d.bidir_fuse(wa, wb, mf, mb))
            return outs

        def fused():
            return d.bidirectional_pyramid([tuple(lv) for lv in levels], holes=False)

        got = {}
        for nm, fn in (("composed", composed), ("fused", fused)):
            def step(fn=fn):
                for t in leaves:
                    t.grad = None
                outs = fn()
                torch.autograd.backward(outs, gouts)
            step()
            got[nm] = [t.grad.clone() for t in leaves]
            before = d.launch_count()
            step()
            torch.cuda.synchronize()
            res[f"residue_mc_{nm}_launches_fwd_bwd"] = d.launch_count() - before
            res[f"residue_mc_{nm}_eager_us"] = time_eager(torch, step)
        res["residue_mc_max_rel_grad_diff"] = max(float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))
                                                  for a, b in zip(got["fused"], got["composed"]))
    for key, step in graphs:
        res[key] = time_graph(torch, step)
        if isinstance(res[key], str):
            break
    print("RESULT " + json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", default="build_variants/parent")
    ap.add_argument("--out", default="profiles/r04")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--worker", nargs=2, metavar=("TREE", "LABEL"))
    a = ap.parse_args()
    if a.worker:
        return worker(os.path.abspath(a.worker[0]), a.out, a.worker[1])
    os.makedirs(a.out, exist_ok=True)
    tmp = tempfile.mkdtemp()
    root = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    runs = []
    for r in range(a.rounds):
        for tree, label in ((a.parent, "parent"), (root, "this")):
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--out", tmp, "--worker", tree, label],
                                 capture_output=True, text=True, env=dict(os.environ, PYTHONDONTWRITEBYTECODE="1"))
            line = [l for l in out.stdout.splitlines() if l.startswith("RESULT ")]
            if out.returncode != 0 or not line:
                raise SystemExit(f"worker {label} failed:\n{out.stdout[-3000:]}\n{out.stderr[-3000:]}")
            runs.append(dict(json.loads(line[0][7:]), round=r))
            print(runs[-1], flush=True)
    import torch
    p, t = torch.load(os.path.join(tmp, "parity_parent.pt")), torch.load(os.path.join(tmp, "parity_this.pt"))
    shutil.rmtree(tmp)
    parity = {k: max(float((x - y).abs().max() / y.abs().max().clamp_min(1e-30)) for x, y in zip(t[k], p[k])) for k in p}
    summary = {"gpu": gpu, "shapes": SHAPES, "max_rel_diff_this_vs_parent": parity, "runs": runs,
               "when": time.strftime("%Y-%m-%d %H:%M:%S")}
    for key in sorted({k for r in runs for k in r}):
        if key.endswith("_us"):
            for label in ("parent", "this"):
                vals = sorted(r[key] for r in runs if r["tree"] == label and isinstance(r.get(key), float))
                if vals:
                    summary[f"median_{label}_{key}"] = vals[len(vals) // 2]
    with open(os.path.join(a.out, "pyramid_bwd_live_batch2.json"), "w") as f:
        json.dump(summary, f, indent=1)
    print(json.dumps({k: v for k, v in summary.items() if k != "runs"}, indent=1))


if __name__ == "__main__":
    main()
