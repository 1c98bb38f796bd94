"""The fused backward of the bi-directional conditioning pyramid (dcb_bidir_pyramid_bwd, csrc/pyramid_bwd.cu): gradients of
both feature maps, both flows and both metrics of every level in two launches, against the CPU oracle's autograd and the
single-op composition; the NO_HOLES fusion; both drop-in extractors on it; the raw ABI."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from tests.util import assert_close


@pytest.fixture(scope="module")
def dcb():
    import diffcodec_b200
    return diffcodec_b200


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    oracle.lib()
    return oracle


LIVE = [(2, 160, 64, 64), (2, 160, 32, 32), (2, 320, 16, 16), (2, 640, 8, 8)]     # Bi_Dir_FeatureExtractor, batch 2
RAGGED = [(2, 30, 19, 19), (1, 19, 23, 17), (3, 8, 8, 8)]                         # C no multiple of 4, odd sizes


def _levels(seed, shapes, null_metric_level=None):
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
        levels.append((first, last, ff, fb, mf, mb))
    return levels


def _gouts(levels, dtype, seed=5):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(lv[0].shape, generator=g).to(dtype) for lv in levels]


def _run_gpu(dcb, levels, gouts, dtype, holes=True, want=range(6)):
    """bidirectional_pyramid with gradients: outputs, the masks it used (saved by the node), the six gradients per level."""
    ts = [[None if t is None else t.cuda().to(dtype) for t in lv] for lv in levels]
    for lv in ts:
        for k in want:
            if lv[k] is not None:
                lv[k].requires_grad_(True)
    outs = dcb.bidirectional_pyramid([tuple(lv) for lv in ts], holes=holes)
    saved = outs[0].grad_fn.saved_tensors
    masks = [(saved[12 * l + 10].float().cpu(), saved[12 * l + 11].float().cpu()) for l in range(len(levels))]
    torch.autograd.backward(list(outs), [g.cuda() for g in gouts])
    return [o.detach() for o in outs], masks, [[None if t is None else t.grad for t in lv] for lv in ts]


def _run_oracle(orc, levels, masks, gouts, holes, dtype=torch.float32):
    """oracle.feature_warper x2 + oracle.fuse with the masks the GPU used (no gradient flows through a mask); torch autograd
    on the CPU gives all six gradients (OracleSplatFunc is differentiable in the flow)."""
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


NAMES = ("first", "last", "flow_f", "flow_b", "metric_f", "metric_b")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("holes", [True, False])
@pytest.mark.parametrize("shapes", ["live", "ragged"])
def test_pyramid_bwd_matches_oracle(dcb, orc, shapes, holes, dtype):
    shp = LIVE if shapes == "live" else RAGGED
    levels = _levels(61, shp, null_metric_level=None if shapes == "live" else 2)
    levels = [tuple(None if t is None else t.to(dtype).float() for t in lv) for lv in levels]      # the values the GPU sees
    gouts = _gouts(levels, dtype)
    outs, masks, grads = _run_gpu(dcb, levels, gouts, dtype, holes)
    for lv, (of, ob) in zip(levels, masks):                        # the masks themselves: equal to the oracle's away from the threshold
        same = (orc.compute_mask(lv[2], lv[3]) == of) & (orc.compute_mask(lv[3], lv[2]) == ob)
        assert same.float().mean() > 0.995
    ref_o, ref_g = _run_oracle(orc, levels, masks, [g.float() for g in gouts], holes)
    if dtype == torch.float32:
        _, truth_g = _run_oracle(orc, levels, masks, [g.double() for g in gouts], holes, torch.float64)
    for l, (o, r) in enumerate(zip(outs, ref_o)):
        tol = 1e-5 if dtype == torch.float32 else 2e-2
        assert_close(o.float(), r, tol, f"fused, level {l}, holes={holes}")
        for k, name in enumerate(NAMES):
            if ref_g[l][k] is None:
                assert grads[l][k] is None
                continue
            assert grads[l][k] is not None and grads[l][k].dtype == dtype and grads[l][k].is_contiguous()
            truth = truth_g[l][k] if dtype == torch.float32 else None
            assert_close(grads[l][k].float(), ref_g[l][k], 2e-5 if dtype == torch.float32 else 2e-2,
                         f"grad {name}, level {l} {tuple(levels[l][0].shape)}, holes={holes}", truth=truth)
        assert float(grads[l][2].abs().max()) > 0 and float(grads[l][3].abs().max()) > 0


@pytest.mark.gpu
def test_no_holes_forward_matches_oracle(dcb, orc):
    """DCB_PYRAMID_NO_HOLES on the inference path: oracle.fuse without occ, with the masks and (1 - mask) kept."""
    levels = _levels(62, RAGGED)
    with torch.no_grad():
        dev = [tuple(None if t is None else t.cuda() for t in lv) for lv in levels]
        fused, saved = dcb.extractors._pyramid_forward(dev, dcb._lib.PYRAMID_NO_HOLES, True)
        assert any(bool(((sv[4] + sv[5]) > 1.5).any()) for sv in saved)                 # there are holes to leave alone
        plain = dcb.bidirectional_pyramid(dev, holes=False)
    for lv, f, p, sv in zip(levels, fused, plain, saved):
        of, ob = sv[4].cpu(), sv[5].cpu()
        wa, ca = orc.feature_warper(lv[0], lv[2], lv[4], of)
        wb, cb = orc.feature_warper(lv[1], lv[3], lv[5], ob)
        assert_close(f, orc.fuse(wa, wb, ca, cb), 1e-5, "NO_HOLES fused")
        assert_close(p, f, 1e-5, "NO_HOLES fused, inference path")


def _composition_inputs():
    # the inputs of test_fused_block_equals_composition (seed 17)
    g = torch.Generator().manual_seed(17)
    n, c, r = 2, 48, 32
    first = torch.randn(n, c, r, r, generator=g).cuda(); last = torch.randn(n, c, r, r, generator=g).cuda()
    ff = (torch.randn(n, 2, r, r, generator=g) * 0.6).cuda(); fb = (-ff.cpu() + 0.25 * torch.randn(n, 2, r, r, generator=g)).cuda()
    mf = (torch.randn(n, 1, r, r, generator=g) * 0.5 + 0.1).cuda(); mb = (torch.randn(n, 1, r, r, generator=g) * 0.5 + 0.1).cuda()
    gout = torch.randn(n, c, r, r, generator=g).cuda()
    return (first, last, ff, fb, mf, mb), gout


class _ByInput(torch.nn.Module):
    """A metric "net" that returns a given tensor per input feature map."""
    def __init__(self, table):
        super().__init__()
        self.table = table

    def forward(self, x):
        return self.table[id(x)]


class _Fixed(torch.nn.Module):
    """A metric "net" that returns a given tensor: the warper's metric gradient lands on that tensor."""
    def __init__(self, m):
        super().__init__()
        self.m = m

    def forward(self, x):
        return self.m


@pytest.mark.gpu
@pytest.mark.parametrize("holes", [True, False])
def test_fused_equals_composition_with_flow_gradients(dcb, holes):
    """One fused node (bidirectional_warp_fuse / bidirectional_pyramid(holes=False)) == the single-op composition (masks, two
    differentiable splats, bidir_fuse with or without occ): values and all six gradients, the two flows included."""
    ins, gout = _composition_inputs()

    def run(fused):
        t = [x.clone().requires_grad_(True) for x in ins]
        first, last, ff, fb, mf, mb = t
        if holes:
            warper = dcb.FeatureWarperSoftsplat(with_learnable_metric=True, in_channels=1).cuda()
            warper.metric_net = _ByInput({id(first): mf, id(last): mb})
            if fused:
                out = dcb.bidirectional_warp_fuse(first, last, ff, fb, warper)
            else:
                with dcb.deterministic():                                # forces bidirectional_warp_fuse onto its composition
                    out = dcb.bidirectional_warp_fuse(first, last, ff, fb, warper)
        elif fused:
            out = dcb.bidirectional_pyramid([(first, last, ff, fb, mf, mb)], holes=False)[0]
        else:
            of, ob = dcb.compute_mask(ff, fb), dcb.compute_mask(fb, ff)
            wa, ca = _warper_with(dcb, mf)(first, ff, mask=of)
            wb, cb = _warper_with(dcb, mb)(last, fb, mask=ob)
            out = dcb.bidir_fuse(wa, wb, ca, cb)
        out.backward(gout)
        return out.detach(), [x.grad for x in t]

    (o1, g1), (o2, g2) = run(True), run(False)
    assert_close(o1, o2, 1e-5, f"fused vs composed, holes={holes}")
    for name, x, y in zip(NAMES, g1, g2):
        assert float(y.abs().max()) > 0, name
        assert_close(x, y, 2e-5, f"fused vs composed grad {name}, holes={holes}")


def _warper_with(dcb, metric):
    w = dcb.FeatureWarperSoftsplat(with_learnable_metric=True, in_channels=1).cuda()
    w.metric_net = _Fixed(metric)
    return w


@pytest.mark.gpu
def test_backward_of_four_levels_is_two_launches(dcb):
    levels = _levels(63, LIVE)
    gouts = [g.cuda() for g in _gouts(levels, torch.float32)]
    for attempt in range(2):                                        # the first round allocates the workspaces
        ts = [[t.cuda().requires_grad_(True) for t in lv] for lv in levels]
        outs = dcb.bidirectional_pyramid([tuple(lv) for lv in ts])
        before = dcb.launch_count()
        torch.autograd.backward(outs, gouts)
        launches = dcb.launch_count() - before
    assert launches == 2


@pytest.mark.gpu
def test_gating_null_metrics_and_channels_last(dcb):
    """Only what was asked for is computed, and it equals the full run; NULL-metric levels; channels_last features."""
    levels = _levels(64, RAGGED, null_metric_level=0)
    gouts = _gouts(levels, torch.float32)
    _, _, full = _run_gpu(dcb, levels, gouts, torch.float32)
    for want in ((2, 3), (0, 1), (0, 5)):
        _, _, part = _run_gpu(dcb, levels, gouts, torch.float32, want=want)
        for l in range(len(levels)):
            for k in range(6):
                if k in want and levels[l][k] is not None:
                    assert_close(part[l][k], full[l][k], 1e-5, f"only {want}: grad {NAMES[k]}, level {l}")
                else:
                    assert part[l][k] is None
    ts = [[None if t is None else t.cuda() for t in lv] for lv in levels]
    for lv in ts:
        lv[0] = lv[0].to(memory_format=torch.channels_last).requires_grad_(True)
        lv[1] = lv[1].to(memory_format=torch.channels_last).requires_grad_(True)
        for k in (2, 3):
            lv[k].requires_grad_(True)
    outs = dcb.bidirectional_pyramid([tuple(lv) for lv in ts])
    torch.autograd.backward(outs, [g.cuda() for g in gouts])
    for l, lv in enumerate(ts):
        for k in range(4):
            assert_close(lv[k].grad, full[l][k], 1e-5, f"channels_last grad {NAMES[k]}, level {l}")


@pytest.mark.gpu
def test_backward_is_bit_identical_run_to_run(dcb):
    levels = _levels(65, LIVE)
    gouts = _gouts(levels, torch.float32)
    ts = [[t.cuda().requires_grad_(True) for t in lv] for lv in levels]
    outs = dcb.bidirectional_pyramid([tuple(lv) for lv in ts])
    grads = []
    for _ in range(2):
        grads.append(torch.autograd.grad(outs, [t for lv in ts for t in lv], [g.cuda() for g in gouts], retain_graph=True))
    for a, b in zip(*grads):
        assert torch.equal(a, b)


def _raw_call(dcb, levels, saved, grads, ws, flags=0, n=None, stream=None):
    lib = dcb._lib.lib()
    arr = dcb._lib.pack_pyramid_bwd(levels, saved, grads)
    return lib.dcb_bidir_pyramid_bwd(arr, len(levels) if n is None else n, ws.data_ptr(), ws.numel(), flags,
                                     stream if stream is not None else dcb._lib.stream_ptr(ws.device))


def _raw_setup(dcb, seed):
    levels = _levels(seed, [(2, 48, 32, 32), (2, 96, 16, 16)])
    dev = [tuple(t.cuda() for t in lv) for lv in levels]
    with torch.no_grad():
        _, saved = dcb.extractors._pyramid_forward(dev, 0, True)
    gouts = [g.cuda() for g in _gouts(levels, torch.float32)]
    ins = [(g,) + lv for g, lv in zip(gouts, dev)]
    grads = [tuple(torch.full((lv[0].shape[0], ch) + tuple(lv[0].shape[2:]), float("nan"), device="cuda") for ch in (lv[0].shape[1],) * 2 + (2, 2, 1, 1))
             for lv in dev]
    return ins, saved, grads


@pytest.mark.gpu
def test_raw_call_replays_in_a_cuda_graph(dcb):
    ins, saved, grads = _raw_setup(dcb, 66)
    lib = dcb._lib.lib()
    need = lib.dcb_bidir_pyramid_bwd_workspace_bytes(dcb._lib.pack_pyramid_bwd(ins, saved, grads), len(ins))
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    assert _raw_call(dcb, ins, saved, grads, ws) == 0
    eager = [[t.clone() for t in gr] for gr in grads]
    assert all(bool(torch.isfinite(t).all()) for gr in eager for t in gr)            # fully overwritten
    for gr in grads:
        for t in gr:
            t.fill_(float("nan"))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            rc = _raw_call(dcb, ins, saved, grads, ws, stream=s.cuda_stream)
    assert rc == 0
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip([t for gr in grads for t in gr], [t for gr in eager for t in gr]):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_raw_abi_errors(dcb):
    ins, saved, grads = _raw_setup(dcb, 67)
    R = dcb._lib
    ws = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    assert _raw_call(dcb, ins, saved, grads, ws, flags=R.PYRAMID_NO_MASKS) == R.E_MODE
    assert _raw_call(dcb, ins, saved, grads, ws, flags=16) == R.E_MODE
    assert _raw_call(dcb, ins, saved, grads, ws, n=0) == R.E_LIMIT
    five = ins * 3
    assert _raw_call(dcb, five[:5], saved * 3, grads * 3, ws) == R.E_LIMIT
    small = torch.empty(256, dtype=torch.uint8, device="cuda")
    assert _raw_call(dcb, ins, saved, grads, small) == R.E_WORKSPACE
    no_metric = [(g, f, l, ff, fb, None, mb) for g, f, l, ff, fb, mf, mb in ins]
    assert _raw_call(dcb, no_metric, saved, grads, ws) == R.E_MODE
    assert _raw_call(dcb, ins, saved, grads, ws, flags=R.PYRAMID_NO_HOLES) == 0


def _reference_residue_forward(dcb, m, prev, nxt, flow_fwd, flow_bwd):
    """Bi_Dir_ResidueExtractor.forward of the reference (controlnet/extractors.py:177-205), restated with single-op calls."""
    x_prev, x_next = m.prev_pre(prev), m.next_pre(nxt)
    outs = []
    for i, res in enumerate(m.resolutions):
        x_prev, x_next = m.prev_pyramids[i](x_prev), m.next_pyramids[i](x_next)
        factor = prev.shape[-2] // res
        flow_f = m.flow_refiners[i](F.interpolate(flow_fwd, size=(res, res), mode="bilinear", align_corners=False) / factor)
        flow_b = m.flow_refiners[i](F.interpolate(flow_bwd, size=(res, res), mode="bilinear", align_corners=False) / factor)
        occ_f, occ_b = dcb.compute_mask(flow_f, flow_b), dcb.compute_mask(flow_b, flow_f)
        conf_prev, conf_next = m.warpers[i].metric_net(x_prev), m.warpers[i].metric_net(x_next)
        warped_prev = dcb.softsplat(tenIn=x_prev, tenFlow=flow_f, tenMetric=conf_prev, strMode="soft") * (1 - occ_f)
        warped_next = dcb.softsplat(tenIn=x_next, tenFlow=flow_b, tenMetric=conf_next, strMode="soft") * (1 - occ_b)
        outs.append(m.zero_convs[i](dcb.bidir_fuse(warped_prev, warped_next, conf_prev, conf_next)))
    return outs


def _nonzero_zero_convs(module, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for zc in module.zero_convs:                                # zero-initialised: no gradient would reach anything else
            for p in zc.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * 0.05)


@pytest.mark.gpu
def test_residue_extractor_dropin_with_flow_gradients(dcb):
    torch.manual_seed(0)
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        m = dcb.Bi_Dir_ResidueExtractor([32, 32, 64, 64]).cuda()
        _nonzero_zero_convs(m, 1)
        with torch.no_grad():                                      # refiners near the identity: flows that are not all occluded
            for r in m.flow_refiners:
                r.weight.mul_(0.1)
                r.weight[:, 0, 1, 1] += 1.0
                r.bias.zero_()
        g = torch.Generator().manual_seed(2)
        prev, nxt = torch.rand(1, 3, 512, 512, generator=g).cuda(), torch.rand(1, 3, 512, 512, generator=g).cuda()
        ff = F.avg_pool2d(torch.randn(1, 2, 512, 512, generator=g), 9, stride=1, padding=4) * 40
        fb = (-ff + torch.randn(1, 2, 512, 512, generator=g) * 0.5).cuda()
        ff = ff.cuda()
        gouts = None
        res = []
        for which in ("ours", "reference"):
            m.zero_grad(set_to_none=True)
            a, b = ff.clone().requires_grad_(True), fb.clone().requires_grad_(True)
            outs = m(prev, nxt, a, b) if which == "ours" else _reference_residue_forward(dcb, m, prev, nxt, a, b)
            if gouts is None:
                gg = torch.Generator().manual_seed(3)
                gouts = [torch.randn(o.shape, generator=gg).cuda() for o in outs]
            before = dcb.launch_count()
            torch.autograd.backward(outs, gouts)
            launches = dcb.launch_count() - before
            grads = {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}
            grads["flow_fwd"], grads["flow_bwd"] = a.grad, b.grad
            res.append(([o.detach() for o in outs], grads, launches))
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    (o1, g1, n1), (o2, g2, _) = res
    assert n1 == 2                                                   # the motion compensation of all four scales
    for i, (x, y) in enumerate(zip(o1, o2)):
        assert_close(x, y, 1e-5, f"residue extractor scale {i}")
    assert set(g1) == set(g2)
    assert float(g2["flow_fwd"].abs().max()) > 0 and float(g2["flow_bwd"].abs().max()) > 0
    assert any(float(g2[k].abs().max()) > 0 for k in g2 if k.startswith("flow_refiners"))
    for k in g2:
        assert_close(g1[k], g2[k], 1e-4, f"residue extractor grad {k}")
    assert list(m.state_dict().keys()) == list(dcb.Bi_Dir_ResidueExtractor([32, 32, 64, 64]).state_dict().keys())


@pytest.mark.gpu
def test_feature_extractor_with_flow_gradients(dcb):
    """flow.requires_grad keeps the whole-pyramid path (differentiable resizes) and matches the scale-by-scale path."""
    torch.manual_seed(0)
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        m = dcb.Bi_Dir_FeatureExtractor([32, 32, 64, 64]).cuda()
        _nonzero_zero_convs(m, 4)
        g = torch.Generator().manual_seed(5)
        cond = torch.rand(1, 6, 512, 512, generator=g).cuda()
        flow = (F.avg_pool2d(torch.randn(1, 4, 512, 512, generator=g), 9, stride=1, padding=4) * 40).cuda()
        gouts = [torch.randn(1, c, r, r, generator=g).cuda() for c, r in zip((32, 32, 64, 64), (64, 32, 16, 8))]
        res = []
        for scale_by_scale in (False, True):
            m.zero_grad(set_to_none=True)
            fl = flow.clone().requires_grad_(True)
            with dcb.deterministic(scale_by_scale):
                before = dcb.launch_count()
                outs = m(cond, fl)
                launches = dcb.launch_count() - before
            torch.autograd.backward(outs, gouts)
            grads = {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}
            grads["flow"] = fl.grad
            res.append(([o.detach() for o in outs], grads, launches))
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    (o1, g1, n1), (o2, g2, n2) = res
    assert n1 == 2 and n2 > n1
    for i, (x, y) in enumerate(zip(o1, o2)):
        assert_close(x, y, 1e-5, f"feature extractor scale {i}")
    assert float(g1["flow"].abs().max()) > 0
    assert set(g1) == set(g2)
    for k in g2:
        assert_close(g1[k], g2[k], 1e-4, f"feature extractor grad {k}")


# ---------------------------------------------------------------------------------------------
# CPU: the workspace query and the argument checks read descriptors only (fake device addresses, nothing is launched)
# ---------------------------------------------------------------------------------------------
def _fake_levels(shapes, metric=True):
    from diffcodec_b200 import _lib
    descs, keep = [], []
    addr = 1 << 32

    def d(n, c, h, w):
        nonlocal addr
        b = ctypes.create_string_buffer(_lib._DESC_STRUCT.pack(addr, _lib.DCB_F32, 0, n, c, h, w, c * h * w, h * w, w, 1))
        addr += 1 << 28
        keep.append(b)
        return ctypes.addressof(b)

    buf = ctypes.create_string_buffer(_lib._BWD_LEVEL_STRUCT.size * max(len(shapes), 1))
    for l, (n, c, h, w) in enumerate(shapes):
        ptrs = [d(n, c, h, w), d(n, c, h, w), d(n, c, h, w), d(n, 2, h, w), d(n, 2, h, w),
                d(n, 1, h, w) if metric else 0, d(n, 1, h, w) if metric else 0]
        ptrs += [addr + 4096 * (i + 1) for i in range(6)]            # saved forward outputs
        ptrs += [addr + (1 << 24) + 4096 * i for i in range(6)]      # gradients
        addr += 1 << 26
        _lib._BWD_LEVEL_STRUCT.pack_into(buf, l * _lib._BWD_LEVEL_STRUCT.size, *ptrs)
    keep.append(buf)
    return ctypes.addressof(buf), keep


def test_workspace_query_and_argument_checks_cpu():
    from diffcodec_b200 import _lib
    lib = _lib.lib()
    shapes = [(2, 160, 64, 64), (2, 160, 32, 32), (2, 320, 16, 16), (2, 640, 8, 8)]
    arr, keep = _fake_levels(shapes)
    want = sum((n * h * w * 24 + 255) // 256 * 256 for n, _, h, w in shapes)
    assert lib.dcb_bidir_pyramid_bwd_workspace_bytes(arr, 4) == want == 2 * 24 * (64 * 64 + 32 * 32 + 16 * 16 + 8 * 8)
    assert lib.dcb_bidir_pyramid_bwd_workspace_bytes(arr, 1) == 2 * 64 * 64 * 24
    odd, keep2 = _fake_levels([(1, 30, 19, 23)])
    assert lib.dcb_bidir_pyramid_bwd_workspace_bytes(odd, 1) == (19 * 23 * 24 + 255) // 256 * 256
    for bad in ((arr, 0), (arr, 5), (arr, -1), (None, 1)):
        assert lib.dcb_bidir_pyramid_bwd_workspace_bytes(*bad) == 0
    # argument errors are found before anything reaches the device
    ws, big = 1 << 40, 1 << 30
    assert lib.dcb_bidir_pyramid_bwd(arr, 4, ws, big, _lib.PYRAMID_NO_MASKS, None) == _lib.E_MODE
    assert lib.dcb_bidir_pyramid_bwd(arr, 4, ws, big, 1, None) == _lib.E_MODE
    assert lib.dcb_bidir_pyramid_bwd(arr, 0, ws, big, 0, None) == _lib.E_LIMIT
    assert lib.dcb_bidir_pyramid_bwd(arr, 5, ws, big, 0, None) == _lib.E_LIMIT
    assert lib.dcb_bidir_pyramid_bwd(None, 1, ws, big, 0, None) == _lib.E_NULL
    assert lib.dcb_bidir_pyramid_bwd(arr, 4, ws, want - 1, 0, None) == _lib.E_WORKSPACE
    assert lib.dcb_bidir_pyramid_bwd(arr, 4, ws + 16, big, 0, None) == _lib.E_WORKSPACE
    nometric, keep3 = _fake_levels(shapes[:1], metric=False)
    assert lib.dcb_bidir_pyramid_bwd(nometric, 1, ws, big, 0, None) == _lib.E_MODE
