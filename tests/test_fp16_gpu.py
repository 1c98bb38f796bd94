"""float16 on the conditioning path: the splat (every forward family, the backward, the deterministic mode), the bi-directional
fusion, the whole-pyramid forward and backward, the batched resampling, the tile merge and both drop-in extractors.

fp16 follows the bf16 rule: loads widened to fp32, fp32 arithmetic, one rounding at each store. The reference of every
check is the CPU oracle run in fp32 on the fp16-rounded inputs; the fp64 oracle is passed as `truth` where the bf16 / fp32
tests pass one. An output is one fp16 rounding (2^-11 = 4.9e-4 relative): 1e-3 for outputs, 2e-3 for gradients (they read
the rounded forward outputs)."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from tests.util import assert_close, make_inputs, oracle_run, cuda_run

OUT_TOL, GRAD_TOL = 1e-3, 2e-3
H = torch.float16


@pytest.fixture(scope="module")
def dcb():
    import diffcodec_b200
    return diffcodec_b200


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    oracle.lib()
    return oracle


MODES = ["sum", "avg", "linear", "soft", "linear-zeroeps", "linear-clipeps", "soft-zeroeps", "soft-clipeps", "soft-addeps"]
# one shape per forward family (csrc/splat_fwd.cu): the accumulator pipeline (a 3-channel frame, and a ragged one), the
# single-launch cluster kernel of small frames, the channel-quad planar pipeline
FAMILY_SHAPES = {"pipe": (2, 3, 96, 128), "pipe_ragged": (3, 3, 97, 131), "small": (2, 3, 24, 40), "planar": (2, 64, 40, 56)}
C4 = (8, 64, 256, 256)                                                   # the per-target list path


def _inputs16(seed, shape, mode, flow_scale=0.4):
    """fp16 inputs and their fp32 values. Flows below half a pixel keep every normaliser O(1): a tiny normaliser amplifies
    the rounding of the saved output by 1/D in the gradients, for the reference as for us (as in the bf16 tests)."""
    tin, flow, metric, gout = make_inputs(seed, *shape, flow_scale=flow_scale)
    if mode.startswith("linear"):
        metric = metric.abs() + 0.25
    return tuple(t.to(H) for t in (tin, flow, metric, gout))


def _close16(got, ref, tol, what, truth=None):
    """assert_close for an fp16 result: where the exact value lies beyond the fp16 range the result is +-inf (rounded once,
    not clamped, as a torch fp16 op gives); everything else within `tol`."""
    g = got.detach().float().cpu()
    r = ref.detach().float().cpu()
    over = torch.isinf(g) & torch.isfinite(r)
    assert bool((r[over].abs() >= 65504.0 * (1 - 1e-3)).all() and (torch.sign(g[over]) == torch.sign(r[over])).all()), what
    assert_close(torch.where(over, r, g), r, tol, what, truth=truth)


def _check_splat(dcb, orc, t16, mode, what, flow=None):
    tin, flow16, metric, gout = t16
    fl = flow16 if flow is None else flow
    ref = oracle_run(orc, tin.float(), fl.float(), metric.float(), gout.float(), mode)
    truth = oracle_run(orc, tin.double(), fl.double(), metric.double(), gout.double(), mode)
    got = cuda_run(dcb.softsplat, tin, fl, metric, gout, mode)
    assert got["out"].dtype == H and got["gin"].dtype == H and got["gflow"].dtype == fl.dtype
    for k in ("out", "gin", "gflow", "gmetric"):
        if ref[k] is not None:
            _close16(got[k], ref[k], OUT_TOL if k == "out" else GRAD_TOL, f"fp16 {what} {mode} {k}", truth=truth[k])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("family", sorted(FAMILY_SHAPES))
def test_softsplat_fp16_matches_oracle(dcb, orc, family, mode):
    _check_splat(dcb, orc, _inputs16(101, FAMILY_SHAPES[family], mode), mode, family)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["sum", "avg", "linear", "soft"])
@pytest.mark.parametrize("family", ["pipe", "small", "planar"])
def test_softsplat_fp16_data_fp32_flow(dcb, orc, family, mode):
    """fp16 data next to an fp32 flow (kept as it is, like bf16): the flow gradient is fp32."""
    t16 = _inputs16(102, FAMILY_SHAPES[family], mode)
    flow32 = make_inputs(103, *FAMILY_SHAPES[family], flow_scale=0.4)[1]
    _check_splat(dcb, orc, t16, mode, f"{family} fp32 flow", flow=flow32)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_softsplat_fp16_list_path(dcb, orc, mode):
    """8 x 64 x 256 x 256 takes the per-target lists, NCHW and channels_last (the channel-quad gather)."""
    lib = dcb._lib.lib()
    n, c, h, w = C4
    m = dcb._lib.MODE_SUM if mode == "sum" else {"avg": 1, "linear": 2, "soft": 3}[mode.split("-")[0]]
    assert lib.dcb_splat_fwd_workspace_is_scratch(n, c, h, w, dcb._lib.DCB_F16, m, 0) == 1
    tin, flow, metric, gout = _inputs16(104, C4, mode)
    ref = oracle_run(orc, tin.float(), flow.float(), metric.float(), gout.float(), mode)
    for layout in (torch.contiguous_format, torch.channels_last):
        x = tin.cuda().to(memory_format=layout)
        before = dcb.launch_count()
        got = cuda_run(dcb.softsplat, x, flow, metric, gout, mode)
        assert got["out"].dtype == H
        _close16(got["out"], ref["out"], OUT_TOL, f"lists {layout} {mode} out")
        for k in ("gin", "gflow", "gmetric"):          # a target that only a far corner reaches: a flow gradient beyond 65504
            if ref[k] is not None:
                _close16(got[k], ref[k], GRAD_TOL, f"lists {layout} {mode} {k}")
        assert dcb.launch_count() - before >= 4


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_deterministic_fp16_is_rounded_fp32(dcb, mode):
    """The deterministic forward is exact in fp32; fp16 is one rounding of that same result, bit for bit."""
    tin, flow, metric, _ = _inputs16(105, (2, 5, 31, 45), mode, flow_scale=4.0)
    me = metric.cuda() if mode.split("-")[0] in ("linear", "soft") else None
    with dcb.deterministic(True):
        a = dcb.softsplat(tin.cuda(), flow.cuda(), me, mode)
        b = dcb.softsplat(tin.cuda().float(), flow.cuda().float(), None if me is None else me.float(), mode)
    assert a.dtype == H
    assert torch.equal(a, b.half())


# ---------------------------------------------------------------------------------------------
# the bi-directional fusion, the pyramid forward and backward
# ---------------------------------------------------------------------------------------------
LIVE = [(2, 160, 64, 64), (2, 160, 32, 32), (2, 320, 16, 16), (2, 640, 8, 8)]     # Bi_Dir_FeatureExtractor, batch 2
RAGGED = [(2, 30, 19, 19), (1, 19, 23, 17), (3, 8, 8, 8)]                         # C no multiple of 4, odd sizes
NAMES = ("first", "last", "flow_f", "flow_b", "metric_f", "metric_b")


def _levels(seed, shapes, null_metric_level=None):
    """Pyramid inputs, already fp16-representable (fp32 tensors holding fp16 values)."""
    g = torch.Generator().manual_seed(seed)
    levels = []
    for l, (n, c, h, w) in enumerate(shapes):
        first, last = torch.randn(n, c, h, w, generator=g), torch.randn(n, c, h, w, generator=g)
        ff = torch.randn(n, 2, h, w, generator=g) * 0.6
        fb = -ff + 0.25 * torch.randn(n, 2, h, w, generator=g)
        mf = torch.randn(n, 1, h, w, generator=g) * 0.5 + 0.1
        mb = torch.randn(n, 1, h, w, generator=g) * 0.5 + 0.1
        if l == null_metric_level:
            mf = mb = None
        levels.append(tuple(None if t is None else t.half().float() for t in (first, last, ff, fb, mf, mb)))
    return levels


def _gouts(levels, seed=5):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(lv[0].shape, generator=g).half() for lv in levels]


def _run_gpu(dcb, levels, gouts, holes=True):
    ts = [[None if t is None else t.cuda().half().requires_grad_(True) for t in lv] for lv in levels]
    outs = dcb.bidirectional_pyramid([tuple(lv) for lv in ts], holes=holes)
    saved = outs[0].grad_fn.saved_tensors
    masks = [(saved[12 * l + 10].float().cpu(), saved[12 * l + 11].float().cpu()) for l in range(len(levels))]
    torch.autograd.backward(list(outs), [g.cuda() for g in gouts])
    return [o.detach() for o in outs], masks, [[None if t is None else t.grad for t in lv] for lv in ts]


def _run_oracle(orc, levels, masks, gouts, holes, dtype=torch.float32):
    outs, grads = [], []
    for lv, (of, ob), go in zip(levels, masks, gouts):
        ts = [None if t is None else t.to(dtype).clone().requires_grad_(True) for t in lv]
        first, last, ff, fb, mf, mb = ts
        wa, ca = orc.feature_warper(first, ff, mf, of.to(dtype))
        wb, cb = orc.feature_warper(last, fb, mb, ob.to(dtype))
        out = orc.fuse(wa, wb, ca, cb, of.to(dtype) if holes else None, ob.to(dtype) if holes else None)
        out.backward(go.to(dtype))
        outs.append(out.detach())
        grads.append([None if t is None else t.grad for t in ts])
    return outs, grads


@pytest.mark.gpu
@pytest.mark.parametrize("holes", [True, False])
@pytest.mark.parametrize("shapes", ["live", "ragged"])
def test_pyramid_fp16_matches_oracle(dcb, orc, shapes, holes):
    levels = _levels(161, LIVE if shapes == "live" else RAGGED, null_metric_level=None if shapes == "live" else 2)
    gouts = _gouts(levels)
    outs, masks, grads = _run_gpu(dcb, levels, gouts, holes)
    for lv, (of, ob) in zip(levels, masks):
        same = (orc.compute_mask(lv[2], lv[3]) == of) & (orc.compute_mask(lv[3], lv[2]) == ob)
        assert same.float().mean() > 0.995
    ref_o, ref_g = _run_oracle(orc, levels, masks, [g.float() for g in gouts], holes)
    _, truth_g = _run_oracle(orc, levels, masks, [g.double() for g in gouts], holes, torch.float64)
    for l, (o, r) in enumerate(zip(outs, ref_o)):
        assert o.dtype == H
        assert_close(o.float(), r, OUT_TOL, f"fused, level {l}, holes={holes}")
        for k, name in enumerate(NAMES):
            if ref_g[l][k] is None:
                assert grads[l][k] is None
                continue
            assert grads[l][k].dtype == H and grads[l][k].is_contiguous()
            assert_close(grads[l][k].float(), ref_g[l][k], GRAD_TOL, f"grad {name}, level {l}, holes={holes}", truth=truth_g[l][k])


@pytest.mark.gpu
def test_pyramid_fp16_launches_determinism_and_graph(dcb):
    """Two launches each way; the backward is bit-identical run to run; forward + backward capture into a CUDA graph and
    replay to the eager values."""
    levels = _levels(162, LIVE)
    gouts = [g.cuda() for g in _gouts(levels)]
    ts = [[t.cuda().half().requires_grad_(True) for t in lv] for lv in levels]
    flat = [t for lv in ts for t in lv]
    for _ in range(2):                                               # the first round allocates the workspaces
        before = dcb.launch_count()
        outs = dcb.bidirectional_pyramid([tuple(lv) for lv in ts])
        fwd = dcb.launch_count() - before
        g1 = torch.autograd.grad(outs, flat, gouts, retain_graph=True)
        bwd = dcb.launch_count() - before - fwd
    assert fwd == 2 and bwd == 2
    g2 = torch.autograd.grad(outs, flat, gouts)
    for a, b in zip(g1, g2):
        assert torch.equal(a, b)

    gts = [[t.detach().clone().requires_grad_(True) for t in lv] for lv in ts]
    gflat = [t for lv in gts for t in lv]

    def step():
        for t in gflat:
            t.grad = None
        outs = dcb.bidirectional_pyramid([tuple(lv) for lv in gts])
        torch.autograd.backward(outs, gouts)
        return outs

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                                       # warm-up on the capture stream
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        g_outs = step()
    graph.replay()
    torch.cuda.synchronize()
    # the forward adds with L2 reductions (last fp32 bits vary), so the replay is compared with the tolerance, not bitwise
    for a, b in zip(g_outs, outs):
        assert_close(a.float(), b.detach().float(), OUT_TOL, "graph replay: fused")
    for t, b in zip(gflat, g1):
        assert_close(t.grad.float(), b.float(), GRAD_TOL, "graph replay: gradient")


@pytest.mark.gpu
def test_pyramid_fp16_no_masks(dcb, orc):
    """DCB_PYRAMID_NO_MASKS (pyramid_conditioning): both soft splats with the all-ones metric, soft_fuse with identity masks."""
    levels = [lv[:4] + (None, None) for lv in _levels(163, [(2, 3, 64, 64), (2, 3, 32, 32), (2, 3, 17, 23)])]
    with torch.no_grad():
        dev = [tuple(None if t is None else t.cuda().half() for t in lv) for lv in levels]
        fused, saved = dcb.extractors._pyramid_forward(dev, dcb._lib.PYRAMID_NO_MASKS, False, want_warped=True)
    for lv, f, sv in zip(levels, fused, saved):
        ones = torch.ones_like(lv[0][:, :1])
        w1, w2 = orc.softsplat(lv[0], lv[2], ones, "soft"), orc.softsplat(lv[1], lv[3], ones, "soft")
        assert f.dtype == H and sv[0].dtype == H
        assert_close(sv[0].float(), w1, OUT_TOL, "NO_MASKS warped1")
        assert_close(sv[1].float(), w2, OUT_TOL, "NO_MASKS warped2")
        assert_close(f.float(), orc.soft_fuse(w1, w2, ones, ones), OUT_TOL, "NO_MASKS fused")
    img = torch.rand(2, 3, 96, 96).cuda().half()
    flow = (torch.randn(2, 2, 96, 96) * 2).cuda().half()
    for w1, w2, f in dcb.pyramid_conditioning(img, img, flow, -flow, sizes=(64, 32)):
        assert f.dtype == H and bool(torch.isfinite(f).all())


@pytest.mark.gpu
def test_bidirectional_block_fp16(dcb, orc):
    """The one-level block through bidirectional_block: forward and all six gradients against the oracle."""
    levels = _levels(164, [(2, 48, 32, 32)])
    gouts = _gouts(levels)
    ts = [t.cuda().half().requires_grad_(True) for t in levels[0]]
    out = dcb.bidirectional_block(*ts)
    saved = out.grad_fn.saved_tensors
    masks = [(saved[10].float().cpu(), saved[11].float().cpu())]
    out.backward(gouts[0].cuda())
    ref_o, ref_g = _run_oracle(orc, levels, masks, [gouts[0].float()], True)
    _, truth_g = _run_oracle(orc, levels, masks, [gouts[0].double()], True, torch.float64)
    assert out.dtype == H
    assert_close(out.detach().float(), ref_o[0], OUT_TOL, "block fused")
    for k, name in enumerate(NAMES):
        assert_close(ts[k].grad.float(), ref_g[0][k], GRAD_TOL, f"block grad {name}", truth=truth_g[0][k])
    with torch.no_grad():                                            # inference path: the same values
        assert_close(dcb.bidirectional_block(*[t.detach() for t in ts]).float(), out.detach().float(), OUT_TOL, "block, inference path")


@pytest.mark.gpu
def test_bidir_fuse_fp16(dcb, orc):
    g = torch.Generator().manual_seed(165)
    n, c, h, w = 2, 19, 21, 27
    vals = [torch.randn(n, c, h, w, generator=g), torch.randn(n, c, h, w, generator=g),
            torch.rand(n, 1, h, w, generator=g) - 0.2, torch.rand(n, 1, h, w, generator=g) - 0.2]
    occ = [(torch.rand(n, 1, h, w, generator=g) > 0.5).float() for _ in range(2)]
    gout = torch.randn(n, c, h, w, generator=g).half()
    vals = [v.half() for v in vals]
    ts = [v.cuda().requires_grad_(True) for v in vals]
    out = dcb.bidir_fuse(*ts, *(o.cuda().half() for o in occ))
    out.backward(gout.cuda())
    rs = [v.float().requires_grad_(True) for v in vals]
    ref = orc.fuse(*rs, *occ)
    ref.backward(gout.float())
    assert out.dtype == H
    assert_close(out.detach().float(), ref.detach(), OUT_TOL, "bidir_fuse fp16")
    for name, t, r in zip(("A", "B", "conf_a", "conf_b"), ts, rs):
        assert t.grad.dtype == H
        assert_close(t.grad.float(), r.grad, GRAD_TOL, f"bidir_fuse fp16 grad {name}")


@pytest.mark.gpu
def test_resample_batch_fp16(dcb):
    """fp16 sources and destinations in any mix with fp32 / bf16, one launch, against F.interpolate on the upcast tensors."""
    g = torch.Generator().manual_seed(166)
    src16 = torch.randn(2, 5, 37, 53, generator=g).cuda().half()
    srcbf = torch.randn(1, 2, 40, 40, generator=g).cuda().bfloat16()
    src32 = torch.randn(2, 2, 64, 64, generator=g).cuda()
    R = dcb._lib
    jobs = [(src16, (16, 24), False, R.RESAMPLE_NONE, 1.0, 1.0), (src16, (50, 70), True, R.RESAMPLE_MUL, 2.0, 0.5, torch.float32),
            (src32, (31, 31), False, R.RESAMPLE_DIV, 15.0, 15.0, H), (srcbf, (8, 8), False, R.RESAMPLE_NONE, 1.0, 1.0, H),
            (src16, (9, 11), False, R.RESAMPLE_NONE, 1.0, 1.0, torch.bfloat16)]
    before = dcb.launch_count()
    outs = dcb.extractors.resample_batch(jobs)
    assert dcb.launch_count() - before == 1
    for (src, size, align, op, f0, f1, *dt), got in zip(jobs, outs):
        want = F.interpolate(src.float(), size=size, mode="bilinear", align_corners=align)
        if op == R.RESAMPLE_MUL:
            want = torch.cat([want[:, :1] * f0, want[:, 1:] * f1], 1)
        elif op == R.RESAMPLE_DIV:
            want = torch.cat([want[:, :1] / f0, want[:, 1:] / f1], 1)
        assert got.dtype == (dt[0] if dt else src.dtype)
        tol = {torch.float32: 1e-5, H: OUT_TOL, torch.bfloat16: 1e-2}[got.dtype]
        assert_close(got.float(), want, tol, f"resample {tuple(src.shape)} -> {size} {got.dtype}")


@pytest.mark.gpu
def test_tile_merge_fp16_1080p(dcb):
    """The 15-tile layout of a 1080p frame (512-pixel tiles, 5 x 3): fp16 latents merge to the fp32 merge of the same values,
    rounded once."""
    xs, ys = (0, 352, 704, 1056, 1408), (0, 284, 568)
    coords = [(x, x + 512, y, y + 512) for y in ys for x in xs]                     # read as (x1, x2, y1, y2)
    g = torch.Generator().manual_seed(167)
    lat = [torch.randn(1, 4, 64, 64, generator=g).half().cuda() for _ in coords]
    got = dcb.merge_latent_tiles_from_pixel_coords(lat, coords, (1, 4, 135, 240), (1080, 1920))
    want = dcb.merge_latent_tiles_from_pixel_coords([t.float() for t in lat], coords, (1, 4, 135, 240), (1080, 1920))
    assert got.dtype == H
    assert torch.equal(got, want.half())


# ---------------------------------------------------------------------------------------------
# the drop-in extractors and the composed builders
# ---------------------------------------------------------------------------------------------
def _nonzero_zero_convs(module, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for zc in module.zero_convs:                                # zero-initialised: no gradient would reach anything else
            for p in zc.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * 0.05)


def _smooth_flow(g, c, scale):
    return F.avg_pool2d(torch.randn(1, c, 512, 512, generator=g), 9, stride=1, padding=4) * scale


@pytest.mark.gpu
def test_feature_extractor_half_model_inference(dcb):
    """An fp16 model (`.half()`) on fp16 inputs: one resample launch and two pyramid launches, fp16 finite outputs."""
    torch.manual_seed(0)
    m = dcb.Bi_Dir_FeatureExtractor([32, 32, 64, 64]).cuda().half()
    _nonzero_zero_convs(m, 6)
    g = torch.Generator().manual_seed(168)
    cond = torch.rand(1, 6, 512, 512, generator=g).cuda().half()
    flow = _smooth_flow(g, 4, 40).cuda().half()
    with torch.no_grad():
        m(cond, flow)                                                # allocates the workspaces
        before = dcb.launch_count()
        outs = m(cond, flow)
        launches = dcb.launch_count() - before
    assert launches == 3
    for o in outs:
        assert o.dtype == H and bool(torch.isfinite(o).all())
    assert float(outs[0].abs().max()) > 0


@pytest.mark.gpu
def test_extractors_under_fp16_autocast(dcb):
    """Training step under torch.autocast(float16): the fp16 feature maps go to the library as they are (one call each way
    for the motion compensation of all four scales), and every warper and refiner parameter gets a finite gradient."""
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(169)
    fe = dcb.Bi_Dir_FeatureExtractor([32, 32, 64, 64]).cuda()
    _nonzero_zero_convs(fe, 7)
    cond = torch.rand(1, 6, 512, 512, generator=g).cuda()
    flow = _smooth_flow(g, 4, 40).cuda()
    re = dcb.Bi_Dir_ResidueExtractor([32, 32, 64, 64]).cuda()
    _nonzero_zero_convs(re, 8)
    with torch.no_grad():                                           # refiners near the identity: flows that are not all occluded
        for r in re.flow_refiners:
            r.weight.mul_(0.1)
            r.weight[:, 0, 1, 1] += 1.0
            r.bias.zero_()
    prev, nxt = torch.rand(1, 3, 512, 512, generator=g).cuda(), torch.rand(1, 3, 512, 512, generator=g).cuda()
    ff = _smooth_flow(g, 2, 40)
    fb = (-ff + torch.randn(1, 2, 512, 512, generator=g) * 0.5).cuda().requires_grad_(True)
    ff = ff.cuda().requires_grad_(True)
    runs = {"feature": (fe, lambda: fe(cond, flow), (3, 2), ("wrapper",)),
            "residue": (re, lambda: re(prev, nxt, ff, fb), (2, 2), ("warpers", "flow_refiners"))}
    for name, (mod, call, (n_fwd, n_bwd), prefixes) in runs.items():
        for _ in range(2):                                          # the first round allocates the workspaces
            mod.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=torch.float16):
                before = dcb.launch_count()
                outs = call()
                fwd = dcb.launch_count() - before
                loss = sum(o.float().square().mean() for o in outs)
            before = dcb.launch_count()
            loss.backward()
            bwd = dcb.launch_count() - before
        assert (fwd, bwd) == (n_fwd, n_bwd), name
        params = [(k, p) for k, p in mod.named_parameters() if k.startswith(prefixes)]
        assert params
        for k, p in params:
            assert p.grad is not None and bool(torch.isfinite(p.grad).all()), f"{name}: {k}"
        assert any(float(p.grad.abs().max()) > 0 for _, p in params), name
    assert bool(torch.isfinite(ff.grad).all()) and float(ff.grad.abs().max()) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("bidir", [False, True])
def test_composed_builders_fp16(dcb, bidir):
    """residual_conditioning[_bidir] on fp16 inputs take the single-op composition (the fused recipes are F32 / BF16), which
    now runs in fp16; it agrees with the fp32 result on the upcast inputs wherever the occlusion masks agree."""
    g = torch.Generator().manual_seed(170)
    n, c, h, w = 2, 3, 72, 96
    img1, img2, gt = (torch.rand(n, c, h, w, generator=g).half() for _ in range(3))
    f1 = F.avg_pool2d(torch.randn(n, 2, h, w, generator=g), 5, stride=1, padding=2) * 6
    f2 = (-f1 + 0.2 * torch.randn(n, 2, h, w, generator=g))
    f1, f2 = f1.half(), f2.half()

    def run(t):
        if bidir:
            return dcb.residual_conditioning_bidir(*(x.cuda().to(t) for x in (img1, img2, f1, f2, gt)), return_masks=True)
        return dcb.residual_conditioning(*(x.cuda().to(t) for x in (img1, f1, f2, gt)), "wrapper", return_masks=True)

    fused, res, of, ob = run(H)
    fused32, res32, of32, ob32 = run(torch.float32)
    assert fused.dtype == H and res.dtype == H
    agree = (of.float() == of32) & (ob.float() == ob32)
    assert agree.float().mean() > 0.99
    keep = agree.expand_as(fused)
    assert_close(torch.where(keep, fused.float(), fused32), fused32, OUT_TOL, "fused")
    assert_close(torch.where(keep, res.float(), res32), res32, OUT_TOL, "residual")


# ---------------------------------------------------------------------------------------------
# the raw ABI: entries without fp16 kernels refuse F16 before any launch
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refusing_entries_on_device(dcb):
    R = dcb._lib
    lib = R.lib()
    img, fl = torch.zeros(1, 3, 16, 16, dtype=H, device="cuda"), torch.zeros(1, 2, 16, 16, dtype=H, device="cuda")
    out, mask = torch.empty_like(img), torch.empty(1, 1, 16, 16, dtype=H, device="cuda")
    ws = torch.empty(1 << 22, dtype=torch.uint8, device="cuda")
    D, st = R.desc, R.stream_ptr(img.device)
    before = dcb.launch_count()
    assert lib.dcb_backwarp_fwd(D(img), D(fl), None, D(out), None, 0, st) == R.E_DTYPE
    assert lib.dcb_backwarp_bwd(D(img), D(img), D(fl), D(out), None, 0, ws.data_ptr(), ws.numel(), st) == R.E_DTYPE
    assert lib.dcb_occlusion_mask(D(fl), D(fl), D(mask), ws.data_ptr(), ws.numel(), 0, st) == R.E_DTYPE
    assert lib.dcb_residual_fused(D(img), D(fl), D(fl), D(img), D(out), D(torch.empty_like(img)), None, None,
                                  ws.data_ptr(), ws.numel(), R.RECIPE_WRAPPER, 0, st) == R.E_DTYPE
    assert lib.dcb_residual_bidir(D(img), D(img), D(fl), D(fl), D(img), D(out), D(torch.empty_like(img)), None, None,
                                  ws.data_ptr(), ws.numel(), 0, st) == R.E_DTYPE
    assert lib.dcb_flow_resize(D(fl), D(torch.empty(1, 2, 8, 8, dtype=H, device="cuda")), 0, st) == R.E_DTYPE
    assert lib.dcb_flow_resize(D(fl.float()), D(torch.empty(1, 2, 8, 8, dtype=H, device="cuda")), 0, st) == R.E_DTYPE
    torch.cuda.synchronize()
    assert dcb.launch_count() == before
    with pytest.raises(ValueError):
        dcb.backwarp(img, fl)


# ---------------------------------------------------------------------------------------------
# CPU: workspace queries and argument checks read descriptors only (fake device addresses, nothing is launched)
# ---------------------------------------------------------------------------------------------
SHAPE_SPREAD = [(1, 1, 8, 8), (2, 3, 24, 40), (2, 3, 96, 128), (4, 4, 135, 240), (64, 3, 1080, 1920), (2, 64, 40, 56),
                (8, 64, 256, 256), (2, 35, 192, 320), (3, 160, 150, 152), (2, 640, 8, 8), (1, 19, 23, 17)]


def _fake(dtype, n, c, h, w, addr=1 << 32, strides=None):
    from diffcodec_b200 import _lib
    s = strides or (c * h * w, h * w, w, 1)
    return _lib._pack_desc(addr, dtype, 0, n, c, h, w, *s)


def test_workspace_queries_f16_equal_bf16_cpu():
    from diffcodec_b200 import _lib
    lib = _lib.lib()
    F16, BF16 = _lib.DCB_F16, _lib.DCB_BF16
    for n, c, h, w in SHAPE_SPREAD:
        for mode in range(4):
            for flags in (0, _lib.FLAG_DETERMINISTIC):
                if flags and n * h * w * 4 >= 1 << 31:
                    continue
                for q in (lib.dcb_splat_fwd_workspace_bytes, lib.dcb_splat_bwd_workspace_bytes, lib.dcb_splat_workspace_bytes,
                          lib.dcb_splat_fwd_workspace_is_scratch):
                    assert q(n, c, h, w, F16, mode, flags) == q(n, c, h, w, BF16, mode, flags), (q.__name__, n, c, h, w, mode, flags)
        for which in (0, 1, 2):
            assert lib.dcb_bidir_block_workspace_bytes(n, c, h, w, F16, which) == lib.dcb_bidir_block_workspace_bytes(n, c, h, w, BF16, which)
    # the list path at the C4 shape is plain scratch in both formats
    assert lib.dcb_splat_fwd_workspace_is_scratch(8, 64, 256, 256, F16, _lib.MODE_SOFT, 0) == 1
    # the pyramid queries: the same bytes for F16 and BF16 levels
    for dt in (F16, BF16):
        keep = []
        lvl = ctypes.create_string_buffer(_lib._LEVEL_STRUCT.size * 4)
        bwd = ctypes.create_string_buffer(_lib._BWD_LEVEL_STRUCT.size * 4)
        for l, (n, c, h, w) in enumerate([(2, 160, 64, 64), (2, 160, 32, 32), (2, 320, 16, 16), (2, 640, 8, 8)]):
            d = [ctypes.create_string_buffer(_fake(dt, n, ch, h, w, (1 << 32) + (l << 28))) for ch in (c, c, 2, 2, 1, 1)]
            keep += d
            ptrs = [ctypes.addressof(b) for b in d]
            _lib._LEVEL_STRUCT.pack_into(lvl, l * _lib._LEVEL_STRUCT.size, *ptrs, *[(1 << 40) + 4096 * i for i in range(7)])
            _lib._BWD_LEVEL_STRUCT.pack_into(bwd, l * _lib._BWD_LEVEL_STRUCT.size, ptrs[0], *ptrs,
                                             *[(1 << 40) + 4096 * i for i in range(12)])
        got = (lib.dcb_bidir_pyramid_workspace_bytes(ctypes.addressof(lvl), 4), lib.dcb_bidir_pyramid_bwd_workspace_bytes(ctypes.addressof(bwd), 4))
        if dt == F16:
            f16 = got
    assert f16 == got and f16[0] > 0 and f16[1] > 0


def test_argument_checks_f16_cpu():
    from diffcodec_b200 import _lib
    lib = _lib.lib()
    F16, BF16, F32, F64 = _lib.DCB_F16, _lib.DCB_BF16, _lib.DCB_F32, _lib.DCB_F64
    n, c, h, w = 2, 3, 16, 16
    ws = 1 << 40
    a = 1 << 32

    def fwd(t_in, t_flow, t_metric, t_out, t_norm=None):
        return lib.dcb_splat_fwd(t_in, t_flow, t_metric, t_out, t_norm, None, ws, 1 << 30, _lib.MODE_SOFT, 0, 0, None)

    m16 = _fake(F16, n, 1, h, w, a + (3 << 24))
    out16 = _fake(F16, n, c, h, w, a + (4 << 24))
    # F16 mixed with BF16, and F16 data with an F64 flow
    assert fwd(_fake(F16, n, c, h, w, a), _fake(BF16, n, 2, h, w, a + (1 << 24)), m16, out16) == _lib.E_DTYPE
    assert fwd(_fake(F16, n, c, h, w, a), _fake(F64, n, 2, h, w, a + (1 << 24)), m16, out16) == _lib.E_DTYPE
    assert fwd(_fake(F16, n, c, h, w, a), _fake(F16, n, 2, h, w, a + (1 << 24)), _fake(BF16, n, 1, h, w, a + (3 << 24)), out16) == _lib.E_DTYPE
    assert fwd(_fake(F16, n, c, h, w, a), _fake(F16, n, 2, h, w, a + (1 << 24)), m16, _fake(BF16, n, c, h, w, a + (4 << 24))) == _lib.E_DTYPE
    assert fwd(_fake(BF16, n, c, h, w, a), _fake(F16, n, 2, h, w, a + (1 << 24)), _fake(BF16, n, 1, h, w, a + (3 << 24)),
               _fake(BF16, n, c, h, w, a + (4 << 24))) == _lib.E_DTYPE
    # the normaliser stays F32 next to F16 data
    assert fwd(_fake(F16, n, c, h, w, a), _fake(F16, n, 2, h, w, a + (1 << 24)), m16, out16, _fake(F16, n, 1, h, w, a + (5 << 24))) == _lib.E_DTYPE
    # an odd F16 pointer (the element size is 2 bytes, not 4)
    assert fwd(_fake(F16, n, c, h, w, a + 1), _fake(F16, n, 2, h, w, a + (1 << 24)), m16, out16) == _lib.E_ALIGN
    assert fwd(_fake(F16, n, c, h, w, a), _fake(F16, n, 2, h, w, a + (1 << 24)), m16, _fake(F16, n, c, h, w, a + (4 << 24) + 1)) == _lib.E_ALIGN
    odd_level = (_fake(F16, n, c, h, w, a + 1),) + tuple(_fake(F16, n, ch, h, w, a + (k << 24)) for k, ch in ((1, c), (2, 2), (3, 2), (4, 1), (5, 1)))
    keep = [ctypes.create_string_buffer(d) for d in odd_level]
    lvl = ctypes.create_string_buffer(_lib._LEVEL_STRUCT.pack(*[ctypes.addressof(b) for b in keep], *[(1 << 40) + 4096 * i for i in range(7)]))
    assert lib.dcb_bidir_pyramid_fwd(ctypes.addressof(lvl), 1, ws, 1 << 30, 0, None) == _lib.E_ALIGN
    # a 2-byte aligned but not 4-byte aligned F16 output is fine for the argument checks of the fusion (no launch: empty batch)
    e = lambda ch, off: _fake(F16, 0, ch, h, w, a + off)
    assert lib.dcb_bidir_fuse_fwd(e(c, 0), e(c, 2 << 24), e(1, 4 << 24), e(1, 6 << 24), None, None, e(c, (8 << 24) + 2), None) == 0
    # the entries without fp16 kernels refuse F16 before anything reaches the device
    img, fl = _fake(F16, n, c, h, w, a), _fake(F16, n, 2, h, w, a + (1 << 24))
    img32, fl32 = _fake(F32, n, c, h, w, a), _fake(F32, n, 2, h, w, a + (1 << 24))
    o = _fake(F16, n, c, h, w, a + (2 << 24))
    assert lib.dcb_backwarp_fwd(img, fl, None, o, None, 0, None) == _lib.E_DTYPE
    assert lib.dcb_backwarp_fwd(img32, fl, None, _fake(F32, n, c, h, w, a + (2 << 24)), None, 0, None) == _lib.E_DTYPE
    assert lib.dcb_backwarp_bwd(o, img, fl, o, None, 0, ws, 1 << 30, None) == _lib.E_DTYPE
    assert lib.dcb_occlusion_mask(fl, fl, _fake(F16, n, 1, h, w, a + (3 << 24)), ws, 1 << 30, 0, None) == _lib.E_DTYPE
    assert lib.dcb_residual_fused(img, fl, fl, img, o, o, None, None, ws, 1 << 30, _lib.RECIPE_WRAPPER, 0, None) == _lib.E_DTYPE
    assert lib.dcb_residual_bidir(img, img, fl, fl, img, o, o, None, None, ws, 1 << 30, 0, None) == _lib.E_DTYPE
    assert lib.dcb_flow_resize(fl, _fake(F16, n, 2, 8, 8, a + (3 << 24)), 0, None) == _lib.E_DTYPE
    assert lib.dcb_flow_resize(fl32, _fake(F16, n, 2, 8, 8, a + (3 << 24)), 0, None) == _lib.E_DTYPE
    # the tile merge takes an F16 canvas (argument checks only: no tiles, an empty canvas)
    assert lib.dcb_tile_merge(None, None, 0, _fake(F16, 1, 4, 0, 0, a), 1080, 1920, 1e-8, None, 0, None) == 0
    assert lib.dcb_tile_merge(None, None, 0, _fake(F16, 1, 4, 8, 8, a + 1), 1080, 1920, 1e-8, None, 0, None) == _lib.E_ALIGN
