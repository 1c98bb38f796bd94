"""The deterministic conditioning pyramid (dcb_bidir_pyramid_fwd with DCB_FLAG_DETERMINISTIC, csrc/pyramid.cu): in fp32 bit for
bit the composition of the deterministic single ops (compute_mask, the masked soft splat of FeatureWarperSoftsplat,
bidir_fuse); both drop-in extractors on it; reproducibility in every dtype (runs, batch position, CUDA-graph replay); the raw
ABI's workspace query and argument checks on the CPU."""
import ctypes
import importlib

import pytest
import torch
import torch.nn.functional as F

from tests.util import assert_close


@pytest.fixture(scope="module")
def dcb():
    import diffcodec_b200
    return diffcodec_b200


LIVE = [(2, 160, 64, 64), (2, 160, 32, 32), (2, 320, 16, 16), (2, 640, 8, 8)]     # Bi_Dir_FeatureExtractor, batch 2
RAGGED = [(2, 30, 19, 19), (1, 19, 23, 17), (3, 8, 8, 8)]                         # C no multiple of 4, odd sizes
COMPRESSIVE = [(2, 12, 48, 40), (2, 20, 24, 20)]                                  # flows that pull whole regions onto a few targets
SETS = {"live": LIVE, "ragged": RAGGED, "compressive": COMPRESSIVE}


def _levels(seed, shapes, kind="random", null_metric_level=None):
    g = torch.Generator().manual_seed(seed)
    levels = []
    for l, (n, c, h, w) in enumerate(shapes):
        first, last = torch.randn(n, c, h, w, generator=g), torch.randn(n, c, h, w, generator=g)
        ff = torch.randn(n, 2, h, w, generator=g) * 0.6
        if kind == "compressive":                                             # 90 % of the way to one point: long target lists
            ys, xs = torch.meshgrid(torch.arange(h, dtype=torch.float32), torch.arange(w, dtype=torch.float32), indexing="ij")
            ff = 0.9 * torch.stack([w / 3 - xs, h / 2 - ys]).expand(n, 2, h, w) + 0.05 * ff
        fb = -ff + 0.25 * torch.randn(n, 2, h, w, generator=g)
        # non-finite and out-of-frame sources in both flows
        for fl in (ff, fb):
            fl[0, 0, 1, 2] = float("nan"); fl[0, 1, 2, 1] = float("inf"); fl[-1, 0, 3, 3] = float("-inf")
            fl[-1, 1, h - 1, 0] = 1e3; fl[0, 0, 0, w - 1] = -2.5 * w
        mf = torch.randn(n, 1, h, w, generator=g) * 0.5 + 0.1
        mb = torch.randn(n, 1, h, w, generator=g) * 0.5 + 0.1
        if l == null_metric_level:
            mf = mb = None
        levels.append((first, last, ff, fb, mf, mb))
    return levels


def _cuda(levels, dtype=torch.float32):
    return [tuple(None if t is None else t.to(dtype).cuda() for t in lv) for lv in levels]


class _Fixed(torch.nn.Module):
    """A metric "net" that returns a given tensor."""
    def __init__(self, m):
        super().__init__()
        self.m = m

    def forward(self, x):
        return self.m


def _warper(dcb, metric):
    if metric is None:
        return dcb.FeatureWarperSoftsplat(with_learnable_metric=False)        # all-ones metric
    w = dcb.FeatureWarperSoftsplat(with_learnable_metric=True, in_channels=1).cuda()
    w.metric_net = _Fixed(metric)
    return w


def _composition(dcb, lv, holes):
    """One scale from the public single ops, under deterministic(): (fused, warped_f, warped_b, norm_f, norm_b, occ_f, occ_b)."""
    ss = importlib.import_module(dcb.__name__ + ".softsplat")          # the submodule (the package re-exports the function)
    _lib = dcb._lib
    first, last, ff, fb, mf, mb = lv
    of, ob = dcb.compute_mask(ff, fb), dcb.compute_mask(fb, ff)
    wa, ca = _warper(dcb, mf)(first, ff, mask=of)
    wb, cb = _warper(dcb, mb)(last, fb, mask=ob)
    ones = torch.ones_like(ff[:, :1])
    _, na = ss._forward(first, ff, ones if mf is None else mf, of, _lib.MODE_SOFT, _lib.EPS_ADD, True, True)
    _, nb = ss._forward(last, fb, ones if mb is None else mb, ob, _lib.MODE_SOFT, _lib.EPS_ADD, True, True)
    fused = dcb.bidir_fuse(wa, wb, ca, cb, of, ob) if holes else dcb.bidir_fuse(wa, wb, ca, cb)
    return fused, wa, wb, na, nb, of, ob


NAMES = ("fused", "warped_f", "warped_b", "norm_f", "norm_b", "occ_f", "occ_b")


@pytest.mark.gpu
@pytest.mark.parametrize("holes", [True, False])
@pytest.mark.parametrize("shapes", ["live", "ragged", "compressive"])
def test_fp32_equals_deterministic_composition(dcb, shapes, holes):
    kind = "compressive" if shapes == "compressive" else "random"
    levels = _cuda(_levels(71, SETS[shapes], kind, null_metric_level=None if shapes == "live" else 1))
    flags = 0 if holes else dcb._lib.PYRAMID_NO_HOLES
    with torch.no_grad(), dcb.deterministic():
        fused, saved = dcb.extractors._pyramid_forward(levels, flags, True)
        for l, lv in enumerate(levels):
            ref = _composition(dcb, lv, holes)
            got = (fused[l],) + tuple(saved[l])
            for name, a, b in zip(NAMES, got, ref):
                assert a.dtype == b.dtype and a.shape == b.shape, (name, l)
                assert torch.equal(a, b), f"{shapes} level {l}: {name} differs from the composition"
        public = dcb.bidirectional_pyramid(levels, holes=holes)                # the public entry, inference path
    for a, b in zip(public, fused):
        assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("shapes", ["ragged", "compressive"])
def test_no_masks_equals_deterministic_softsplat_composition(dcb, shapes):
    """DCB_PYRAMID_NO_MASKS: deterministic soft splats with the level's metrics (all-ones where NULL), fused with those
    metrics as confidences, without masks or holes."""
    kind = "compressive" if shapes == "compressive" else "random"
    levels = _cuda(_levels(72, SETS[shapes], kind, null_metric_level=0))
    with torch.no_grad(), dcb.deterministic():
        fused, saved = dcb.extractors._pyramid_forward(levels, dcb._lib.PYRAMID_NO_MASKS, False, want_warped=True)
        for l, (first, last, ff, fb, mf, mb) in enumerate(levels):
            ones = torch.ones_like(ff[:, :1])
            mf, mb = ones if mf is None else mf, ones if mb is None else mb
            wa = dcb.softsplat(tenIn=first, tenFlow=ff, tenMetric=mf, strMode="soft")
            wb = dcb.softsplat(tenIn=last, tenFlow=fb, tenMetric=mb, strMode="soft")
            assert torch.equal(saved[l][0], wa) and torch.equal(saved[l][1], wb), l
            assert torch.equal(fused[l], dcb.bidir_fuse(wa, wb, mf, mb)), l


@pytest.mark.gpu
def test_pyramid_conditioning_equals_composition(dcb):
    g = torch.Generator().manual_seed(73)
    img1, img2 = torch.rand(2, 3, 96, 96, generator=g).cuda(), torch.rand(2, 3, 96, 96, generator=g).cuda()
    flow1 = (F.avg_pool2d(torch.randn(2, 2, 96, 96, generator=g), 7, stride=1, padding=3) * 30).cuda()
    flow2 = -flow1 + torch.randn(2, 2, 96, 96, generator=g).cuda()
    sizes = (64, 32, 16)
    R = dcb._lib
    with torch.no_grad(), dcb.deterministic():
        out = dcb.pyramid_conditioning(img1, img2, flow1, flow2, sizes)
        for (w1, w2, fused), size in zip(out, sizes):
            s = float(size) / float(flow1.shape[-1])
            a, b, f1, f2 = dcb.resample_batch([(img1, (size, size), False, R.RESAMPLE_NONE, 1.0, 1.0), (img2, (size, size), False, R.RESAMPLE_NONE, 1.0, 1.0),
                                               (flow1, (size, size), False, R.RESAMPLE_MUL, s, s), (flow2, (size, size), False, R.RESAMPLE_MUL, s, s)])
            ones = torch.ones_like(f1[:, :1])
            r1 = dcb.softsplat(tenIn=a, tenFlow=f1, tenMetric=ones, strMode="soft")
            r2 = dcb.softsplat(tenIn=b, tenFlow=f2, tenMetric=ones, strMode="soft")
            assert torch.equal(w1, r1) and torch.equal(w2, r2), size
            assert torch.equal(fused, dcb.bidir_fuse(r1, r2, ones, ones)), size


def _nonzero_zero_convs(module, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for zc in module.zero_convs:                                # zero-initialised: no gradient would reach anything else
            for p in zc.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * 0.05)


class _ExactConvs:
    """cuDNN's deterministic algorithms without TF32: the conv outputs of two runs are the same bits."""
    def __enter__(self):
        b = torch.backends
        self.saved = (b.cudnn.deterministic, b.cudnn.benchmark, b.cudnn.allow_tf32, b.cuda.matmul.allow_tf32)
        b.cudnn.deterministic, b.cudnn.benchmark, b.cudnn.allow_tf32, b.cuda.matmul.allow_tf32 = True, False, False, False

    def __exit__(self, *exc):
        b = torch.backends
        b.cudnn.deterministic, b.cudnn.benchmark, b.cudnn.allow_tf32, b.cuda.matmul.allow_tf32 = self.saved
        return False


def _feature_loop(dcb, m, cond, flow):
    """Bi_Dir_FeatureExtractor.forward scale by scale from single ops (controlnet/extractors.py:266-314)."""
    f, l = m.first_pre_extractor(cond[:, 3:]), m.last_pre_extractor(cond[:, :3])
    outs = []
    for idx, res in enumerate((64, 32, 16, 8)):
        f, l = m.extractors_first[idx](f), m.extractors_last[idx](l)
        ff = dcb.resize_and_normalize_flow_batched(flow[:, :2], res, res)
        fb = dcb.resize_and_normalize_flow_batched(flow[:, 2:], res, res)
        of, ob = dcb.compute_mask(ff, fb), dcb.compute_mask(fb, ff)
        wa, ca = m.wrapper[idx](f, ff, mask=of)
        wb, cb = m.wrapper[idx](l, fb, mask=ob)
        outs.append(m.zero_convs[idx](dcb.bidir_fuse(wa, wb, ca, cb, of, ob)))
    return outs


def _residue_loop(dcb, m, prev, nxt, flow_fwd, flow_bwd):
    """Bi_Dir_ResidueExtractor.forward scale by scale from single ops (controlnet/extractors.py:177-205)."""
    x_prev, x_next = m.prev_pre(prev), m.next_pre(nxt)
    outs = []
    for i, res in enumerate(m.resolutions):
        x_prev, x_next = m.prev_pyramids[i](x_prev), m.next_pyramids[i](x_next)
        factor = prev.shape[-2] // res
        ff = m.flow_refiners[i](F.interpolate(flow_fwd, size=(res, res), mode="bilinear", align_corners=False) / factor)
        fb = m.flow_refiners[i](F.interpolate(flow_bwd, size=(res, res), mode="bilinear", align_corners=False) / factor)
        of, ob = dcb.compute_mask(ff, fb), dcb.compute_mask(fb, ff)
        wa, ca = m.warpers[i](x_prev, ff, mask=of)
        wb, cb = m.warpers[i](x_next, fb, mask=ob)
        outs.append(m.zero_convs[i](dcb.bidir_fuse(wa, wb, ca, cb)))
    return outs


def _run_extractor(dcb, m, fn, inputs, gouts):
    """Forward under deterministic() (library launches counted), backward; outputs, parameter + input gradients, launches."""
    m.zero_grad(set_to_none=True)
    ins = [t.clone().requires_grad_(True) for t in inputs]
    with dcb.deterministic():
        before = dcb.launch_count()
        outs = fn(*ins)
        launches = dcb.launch_count() - before
    torch.autograd.backward(outs, gouts)
    grads = {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}
    for i, t in enumerate(ins):
        grads[f"input{i}"] = t.grad
    return [o.detach() for o in outs], grads, launches


def _check_extractor(dcb, m, inputs, loop):
    gg = torch.Generator().manual_seed(3)
    with _ExactConvs():
        with torch.no_grad(), dcb.deterministic():
            shapes = [o.shape for o in m(*inputs)]
        gouts = [torch.randn(s, generator=gg).cuda() for s in shapes]
        o1, g1, n1 = _run_extractor(dcb, m, m, inputs, gouts)
        o2, g2, _ = _run_extractor(dcb, m, m, inputs, gouts)
        o3, g3, n3 = _run_extractor(dcb, m, lambda *t: loop(dcb, m, *t), inputs, gouts)
        with torch.no_grad(), dcb.deterministic():                  # inference: the flows are resized by one library launch
            before = dcb.launch_count()
            o4 = m(*inputs)
            n4 = dcb.launch_count() - before
            o5 = m(*inputs)
    assert n1 <= 12 and n4 <= 12 and n3 > n1, (n1, n4, n3)
    for i, (a, b, c) in enumerate(zip(o1, o2, o3)):
        assert torch.equal(a, c), f"scale {i}: pyramid vs scale-by-scale loop"
        assert torch.equal(a, b), f"scale {i}: run to run"
    for a, b in zip(o4, o5):
        assert torch.equal(a, b)
    assert set(g1) == set(g2) == set(g3)
    for k in g1:
        assert torch.equal(g1[k], g2[k]), f"grad {k}: run to run"
        assert_close(g1[k], g3[k], 1e-4, f"grad {k} vs the composition")
    assert any(float(g3[k].abs().max()) > 0 for k in g3 if k.startswith("input"))


@pytest.mark.gpu
def test_feature_extractor_deterministic_fp32(dcb):
    torch.manual_seed(0)
    m = dcb.Bi_Dir_FeatureExtractor([32, 32, 64, 64]).cuda()
    _nonzero_zero_convs(m, 4)
    g = torch.Generator().manual_seed(5)
    cond = torch.rand(2, 6, 512, 512, generator=g).cuda()
    flow = (F.avg_pool2d(torch.randn(2, 4, 512, 512, generator=g), 9, stride=1, padding=4) * 40).cuda()
    _check_extractor(dcb, m, [cond, flow], _feature_loop)


@pytest.mark.gpu
def test_residue_extractor_deterministic_fp32(dcb):
    torch.manual_seed(0)
    m = dcb.Bi_Dir_ResidueExtractor([32, 32, 64, 64]).cuda()
    _nonzero_zero_convs(m, 1)
    with torch.no_grad():                                          # refiners near the identity: flows that are not all occluded
        for r in m.flow_refiners:
            r.weight.mul_(0.1)
            r.weight[:, 0, 1, 1] += 1.0
            r.bias.zero_()
    g = torch.Generator().manual_seed(2)
    prev, nxt = torch.rand(2, 3, 512, 512, generator=g).cuda(), torch.rand(2, 3, 512, 512, generator=g).cuda()
    ff = F.avg_pool2d(torch.randn(2, 2, 512, 512, generator=g), 9, stride=1, padding=4) * 40
    fb = (-ff + torch.randn(2, 2, 512, 512, generator=g) * 0.5).cuda()
    _check_extractor(dcb, m, [prev, nxt, ff.cuda(), fb], _residue_loop)


@pytest.mark.gpu
def test_block_under_the_flag_is_the_one_level_pyramid(dcb):
    lv = _cuda(_levels(74, [(2, 48, 32, 32)]))[0]
    with torch.no_grad(), dcb.deterministic():
        a = dcb.bidirectional_block(*lv)
        b = _composition(dcb, lv, True)[0]
    assert torch.equal(a, b)


DTYPES = [torch.float32, torch.bfloat16, torch.float16]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_reproducible_runs_and_batch_position(dcb, dtype):
    levels = _levels(75, [(4, c, h, w) for _, c, h, w in LIVE])
    dev = _cuda(levels, dtype)
    with torch.no_grad(), dcb.deterministic():
        runs = [dcb.bidirectional_pyramid(dev) for _ in range(3)]
        for r in runs[1:]:
            for a, b in zip(runs[0], r):
                assert torch.equal(a, b)
        k = 2
        alone = dcb.bidirectional_pyramid([tuple(None if t is None else t[k:k + 1] for t in lv) for lv in dev])
    for a, b in zip(runs[0], alone):
        assert torch.equal(a[k:k + 1], b)
    if dtype != torch.float32:                                      # same inputs in fp32: the cells are the same fp32 sums
        exact = [tuple(None if t is None else t.float() for t in lv) for lv in dev]
        with torch.no_grad(), dcb.deterministic():
            ref = dcb.bidirectional_pyramid(exact)
        for l, (a, b) in enumerate(zip(runs[0], ref)):
            assert_close(a.float(), b, 1e-2, f"{dtype} vs fp32, level {l}")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_raw_call_replays_in_a_cuda_graph(dcb, dtype):
    R = dcb._lib
    lib = R.lib()
    levels = _cuda(_levels(76, RAGGED, null_metric_level=2), dtype)
    outs = []
    for first, *_ in levels:
        n, c, h, w = first.shape
        outs.append((torch.empty_like(first), torch.empty_like(first), torch.empty_like(first),
                     torch.empty((n, 1, h, w), device="cuda"), torch.empty((n, 1, h, w), device="cuda"),
                     torch.empty((n, 1, h, w), dtype=dtype, device="cuda"), torch.empty((n, 1, h, w), dtype=dtype, device="cuda")))
    need = lib.dcb_bidir_pyramid_det_workspace_bytes(R.pack_pyramid(levels, outs), len(levels))
    assert need >= lib.dcb_bidir_pyramid_workspace_bytes(R.pack_pyramid(levels, outs), len(levels))
    ws = torch.full((need,), 0xFF, dtype=torch.uint8, device="cuda")            # plain scratch: any contents

    def call(stream):
        return lib.dcb_bidir_pyramid_fwd(R.pack_pyramid(levels, outs), len(levels), ws.data_ptr(), need, R.FLAG_DETERMINISTIC, stream)

    assert call(R.stream_ptr(ws.device)) == 0
    eager = [[t.clone() for t in o] for o in outs]
    for o in outs:
        for t in o:
            t.fill_(float("nan"))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            rc = call(s.cuda_stream)
    assert rc == 0
    for _ in range(2):
        graph.replay()
    torch.cuda.synchronize()
    for a, b in zip([t for o in outs for t in o], [t for o in eager for t in o]):
        assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------
# CPU: the workspace query and the argument checks read descriptors only (fake device addresses, nothing is launched)
# ---------------------------------------------------------------------------------------------
def _fake_levels(shapes):
    from diffcodec_b200 import _lib
    keep = []
    addr = 1 << 32

    def d(n, c, h, w):
        nonlocal addr
        b = ctypes.create_string_buffer(_lib._DESC_STRUCT.pack(addr, _lib.DCB_F32, 0, n, c, h, w, c * h * w, h * w, w, 1))
        addr += 1 << 36
        keep.append(b)
        return ctypes.addressof(b)

    buf = ctypes.create_string_buffer(_lib._LEVEL_STRUCT.size * len(shapes))
    for l, (n, c, h, w) in enumerate(shapes):
        ptrs = [d(n, c, h, w), d(n, c, h, w), d(n, 2, h, w), d(n, 2, h, w), d(n, 1, h, w), d(n, 1, h, w)]
        ptrs += [addr + (1 << 34) * (i + 1) for i in range(7)]       # fused, warped_*, norm_*, occ_*
        addr += 1 << 38
        _lib._LEVEL_STRUCT.pack_into(buf, l * _lib._LEVEL_STRUCT.size, *ptrs)
    keep.append(buf)
    return ctypes.addressof(buf), keep


def test_det_workspace_query_and_argument_checks_cpu():
    from diffcodec_b200 import _lib
    lib = _lib.lib()
    arr, keep = _fake_levels(LIVE)
    keys = 4 * 2 * sum(n * h * w for n, _, h, w in LIVE)
    plain = lib.dcb_bidir_pyramid_workspace_bytes(arr, 4)
    det = lib.dcb_bidir_pyramid_det_workspace_bytes(arr, 4)
    assert plain > 0 and det >= plain + 2 * 8 * keys                   # keys and sorted keys on top of the cells
    assert lib.dcb_bidir_pyramid_workspace_bytes(arr, 4) == plain      # the plain query is unchanged
    for bad in ((arr, 0), (arr, 5), (arr, -1), (None, 1)):
        assert lib.dcb_bidir_pyramid_det_workspace_bytes(*bad) == 0
    ws, big = 1 << 40, 1 << 40
    DET, CLEAN = _lib.FLAG_DETERMINISTIC, _lib.FLAG_WS_CLEAN
    assert lib.dcb_bidir_pyramid_fwd(arr, 4, ws, big, DET | CLEAN, None) == _lib.E_MODE
    assert lib.dcb_bidir_pyramid_fwd(arr, 4, ws, big, DET | 16, None) == _lib.E_MODE
    assert lib.dcb_bidir_pyramid_fwd(arr, 4, ws, big, 16, None) == _lib.E_MODE
    assert lib.dcb_bidir_pyramid_fwd(arr, 4, ws, big, 32, None) == _lib.E_MODE
    assert lib.dcb_bidir_pyramid_fwd(arr, 4, ws, det - 1, DET, None) == _lib.E_WORKSPACE
    assert lib.dcb_bidir_pyramid_fwd(arr, 4, ws + 16, big, DET | _lib.PYRAMID_NO_HOLES, None) == _lib.E_WORKSPACE
    # 4 keys per pixel, two directions: 8 * 16384 * 16384 = 2^31 keys is one too many; one row less fits
    huge, keep2 = _fake_levels([(1, 1, 16384, 16384)])
    assert lib.dcb_bidir_pyramid_fwd(huge, 1, ws, big, DET, None) == _lib.E_LIMIT
    fits, keep3 = _fake_levels([(1, 1, 16383, 16384)])
    assert lib.dcb_bidir_pyramid_fwd(fits, 1, ws, 256, DET, None) == _lib.E_WORKSPACE
    assert lib.dcb_bidir_pyramid_det_workspace_bytes(fits, 1) > 2 * 8 * 8 * 16383 * 16384
