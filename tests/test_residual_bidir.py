"""The two-reference conditioning builder (residual_conditioning_bidir / dcb_residual_bidir): both I-frames warped by their
own flows, fused by occlusion (soft_fuse on the valid masks, pairing of extractors.py:290-295), subtracted from the ground
truth. CPU: oracle known answers and workspace queries. GPU: parity with the oracle on every forward path, the strided views
of the reference's datasets, the composed fallback, raw ABI errors and CUDA-graph capture."""
import pytest
import torch

from tests.util import assert_close, make_inputs


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    oracle.lib()
    return oracle


def _flows(seed, n, h, w, scale):
    g = torch.Generator().manual_seed(seed)
    f1 = torch.randn(n, 2, h, w, generator=g) * scale
    f1 = torch.nn.functional.avg_pool2d(torch.nn.functional.pad(f1, (2, 2, 2, 2), mode="replicate"), 5, stride=1) * 2
    f2 = -f1 + torch.randn(n, 2, h, w, generator=g) * 0.15 * scale
    return f1, f2


def _recipe_bidir(orc, image1, image2, flow1, flow2, gt):
    """The two-reference recipe on CPU tensors, composed from the oracle's restatements of the reference functions:
    image_k moved by flow_k (softsplat.py:232-274, all-ones metric), occlusion masks with the pairing of extractors.py:290-295
    (control_utils.py:11-17), soft_fuse on the VALID masks (improv_experiments.ipynb cell 3: holes where both references are
    occluded), residual against gt. Returns (fused, residual, occ_fwd, occ_bwd)."""
    ones = torch.ones_like(flow1[:, :1])
    warped1 = orc.softsplat(image1, flow1, ones, "soft")
    warped2 = orc.softsplat(image2, flow2, ones, "soft")
    occ_fwd = orc.compute_mask(flow1, flow2)
    occ_bwd = orc.compute_mask(flow2, flow1)
    fused = orc.soft_fuse(warped1, warped2, 1 - occ_fwd, 1 - occ_bwd)
    return fused, gt - fused, occ_fwd, occ_bwd


def _frames(seed, n, c, h, w):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(n, c, h, w, generator=g), torch.rand(n, c, h, w, generator=g), torch.rand(n, c, h, w, generator=g)


# ---------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------
def test_oracle_zero_flow_is_the_average(orc):
    """No motion: no mask fires, both references are valid, fused = (image1 + image2) / (2 + 1e-6) up to the 1e-7 eps."""
    img1, img2, gt = _frames(1, 2, 3, 12, 16)
    zero = torch.zeros(2, 2, 12, 16)
    fused, res, of, ob = _recipe_bidir(orc, img1, img2, zero, zero, gt)
    assert float(of.abs().max()) == 0 and float(ob.abs().max()) == 0
    assert_close(fused, (img1 + img2) / 2, 2e-6, "zero flow")
    assert_close(res, gt - fused, 0, "residual")


def test_oracle_both_occluded_fills_the_hole(orc):
    """flow2 pushes every pixel of image2 out of the frame: warped2 = 0, both masks fire everywhere, and the hole fill
    gives 0.5 * (warped1 + warped2) = 0.5 * warped1."""
    img1, img2, gt = _frames(2, 1, 3, 10, 14)
    flow1 = torch.zeros(1, 2, 10, 14)
    flow2 = torch.full((1, 2, 10, 14), 1000.0)
    fused, res, of, ob = _recipe_bidir(orc, img1, img2, flow1, flow2, gt)
    assert bool((of == 1).all()) and bool((ob == 1).all())
    warped1 = orc.softsplat(img1, flow1, torch.ones(1, 1, 10, 14), "soft")
    assert_close(fused, 0.5 * warped1, 1e-7, "hole fill")
    assert_close(fused, 0.5 * img1, 1e-6, "hole fill ~ image1 / 2")


def test_workspace_query_serves_the_bidir_entry():
    """dcb_residual_bidir is sized with dcb_residual_workspace_bytes: the rider pipeline slot (float4 + float2 cells of one
    1080p frame) and the two mask planes, without a GPU."""
    import diffcodec_b200
    L = diffcodec_b200._lib
    lib = L.lib()
    hw = 1080 * 1920
    assert lib.dcb_residual_workspace_bytes(1, 3, 1080, 1920) == hw * (24 + 8)
    assert lib.dcb_residual_workspace_bytes(64, 3, 1080, 1920) == hw * 24 + 2 * 64 * hw * 4
    assert lib.dcb_residual_workspace_bytes(3, 1, 1080, 1920) == hw * 24 + 2 * 3 * hw * 4
    assert hasattr(lib, "dcb_residual_bidir") and "dcb_residual_bidir" in L.SYMBOLS


# ---------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dcb():
    import diffcodec_b200
    return diffcodec_b200


def _ru(dcb):
    from importlib import import_module
    return import_module(dcb.__name__ + ".residual_utils")


def _mask_mismatch(got, ref, a, b, orc):
    """Mask entries may legitimately flip only where ||.|| is within fp32 noise of the 0.3 threshold."""
    diff = (got.float().cpu() != ref)
    if not diff.any():
        return 0
    nrm = torch.norm(b + orc.softsplat(a, b, torch.ones_like(b[:, :1]), "soft"), p=2, dim=1, keepdim=True)
    assert ((nrm[diff] - 0.3).abs() < 1e-5).all(), "mask differs away from the threshold"
    return int(diff.sum())


class _Path:
    def __init__(self, dcb, fwd_path, group_frames, h, w):
        self.L, self.fwd_path, self.group_bytes = dcb._lib, fwd_path, group_frames * h * w * 16

    def __enter__(self):
        self.L.set_option("fwd_path", self.fwd_path)
        self.L.set_option("pipe_group_bytes", self.group_bytes)
        self.L.release_workspaces()

    def __exit__(self, *exc):
        self.L.set_option("fwd_path", 0)
        self.L.set_option("pipe_group_bytes", 0)
        self.L.release_workspaces()
        return False


# (fwd_path, shape, frames per pipeline group): default dispatch on small frames (cluster kernels + fusion kernel) and on a
# frame the pipeline takes, the pinned pipeline over several ragged groups, the owner kernels
_CASES = [(0, (2, 3, 64, 64), 0), (0, (2, 3, 96, 120), 0), (1, (5, 3, 33, 47), 2), (1, (3, 1, 70, 150), 1), (1, (4, 2, 45, 64), 3),
          (1, (2, 3, 96, 120), 0), (2, (2, 3, 40, 56), 0), (2, (3, 2, 33, 47), 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("fwd_path,shape,group_frames", _CASES)
def test_bidir_matches_oracle(dcb, orc, fwd_path, shape, group_frames, dtype):
    n, c, h, w = shape
    with _Path(dcb, fwd_path, group_frames, h, w):
        img1, img2, gt = _frames(23, n, c, h, w)
        f1, f2 = _flows(6, n, h, w, 2.0)
        if dtype == torch.bfloat16:
            img1, img2, gt, f1, f2 = (t.bfloat16().float() for t in (img1, img2, gt, f1, f2))
        fused_r, res_r, of_r, ob_r = _recipe_bidir(orc, img1, img2, f1, f2, gt)
        dev = [t.cuda().to(dtype) for t in (img1, img2, f1, f2, gt)]
        l0 = dcb.launch_count()
        fused, res, of, ob = dcb.residual_conditioning_bidir(*dev, return_masks=True)
        launches = dcb.launch_count() - l0
        assert fused.dtype == dtype and fused.shape == (n, c, h, w) and of.shape == (n, 1, h, w)
        if fwd_path == 1 or (fwd_path == 0 and h * w > 8192):
            groups = 1 if group_frames == 0 else -(-n // group_frames)
            assert launches == 4 * groups                 # two passes, each one scatter + one epilogue launch per frame group
        tol = 1e-5 if dtype == torch.float32 else 1.6e-2
        agree = (of.float().cpu() == of_r) & (ob.float().cpu() == ob_r)
        if dtype == torch.float32:
            assert _mask_mismatch(of, of_r, f1, f2, orc) + _mask_mismatch(ob, ob_r, f2, f1, orc) <= 2
        else:
            assert agree.float().mean() >= 0.995
        assert 0 < float(of_r.mean()) < 1 and 0 < float(ob_r.mean()) < 1
        sel = agree.expand_as(fused_r)
        assert_close(fused.float().cpu()[sel], fused_r[sel], tol, "fused")
        assert_close(res.float().cpu()[sel], res_r[sel], tol, "residual")
        if dtype == torch.float32:                        # fused entry == composition of the single-op kernels where the masks agree
            fc, rc_, ofc, obc = _ru(dcb)._composed_bidir(*dev)
            same = ((ofc == of) & (obc == ob)).expand_as(fused)
            assert same.float().mean() > 0.99
            assert_close(fused[same], fc[same], 1e-5, "fused vs composed")
            assert_close(res[same], rc_[same], 1e-5, "residual vs composed")
        # the kept-zero workspace was left all-zero: the next splat through it is right
        tin, flow, metric, _ = make_inputs(3, 2, 3, h, w)
        assert_close(dcb.softsplat(tin.cuda(), flow.cuda(), metric.cuda(), "soft"), orc.softsplat(tin, flow, metric, "soft"), 1e-5,
                     "softsplat after the bidir recipe")


@pytest.mark.gpu
@pytest.mark.parametrize("fwd_path", [0, 1])
@pytest.mark.parametrize("shape", [(3, 3, 96, 120), (3, 3, 33, 47)])
def test_bidir_strided_views(dcb, shape, fwd_path):
    """Channel slices of one 6-channel image tensor and of one [N,4,H,W] flow tensor, a channels_last image, a row-padded gt
    and I-frames given as expanded (stride-0) batches: the same values as the contiguous call."""
    n, c, h, w = shape
    with _Path(dcb, fwd_path, 0, h, w):
        img1, img2, gt = (t.cuda() for t in _frames(29, n, c, h, w))
        f1, f2 = (t.cuda() for t in _flows(8, n, h, w, 2.0))
        ref = dcb.residual_conditioning_bidir(img1, img2, f1, f2, gt, return_masks=True)
        both_img = torch.cat([img1, img2], dim=1)                               # [N,6,H,W]: local_conditions-like
        both_flow = torch.cat([f1, f2], dim=1)                                  # [N,4,H,W]
        gt_pad = torch.zeros(n, c, h, w + 3, device="cuda"); gt_pad[..., :w] = gt
        views = [(both_img[:, :c], both_img[:, c:], both_flow[:, :2], both_flow[:, 2:], gt_pad[..., :w]),
                 (img1.to(memory_format=torch.channels_last), img2, f1, f2, gt)]
        assert not both_img[:, c:].is_contiguous() and not both_flow[:, 2:].is_contiguous() and not gt_pad[..., :w].is_contiguous()
        for args in views:
            got = dcb.residual_conditioning_bidir(*args, return_masks=True)
            assert torch.equal(got[2], ref[2]) and torch.equal(got[3], ref[3])
            assert_close(got[0], ref[0], 2e-6, "fused, strided views")
            assert_close(got[1], ref[1], 2e-6, "residual, strided views")
        # one I-frame pair serving all N inter frames (a GOP): stride-0 batch vs the materialised repeat
        e1, e2 = img1[:1].expand(n, c, h, w), img2[:1].expand(n, c, h, w)
        assert e1.stride(0) == 0
        got = dcb.residual_conditioning_bidir(e1, e2, f1, f2, gt, return_masks=True)
        rep = dcb.residual_conditioning_bidir(e1.contiguous(), e2.contiguous(), f1, f2, gt, return_masks=True)
        assert torch.equal(got[2], rep[2]) and torch.equal(got[3], rep[3])
        assert_close(got[0], rep[0], 2e-6, "fused, expanded I-frames")
        assert_close(got[1], rep[1], 2e-6, "residual, expanded I-frames")


@pytest.mark.gpu
def test_bidir_composed_paths(dcb, orc):
    """More than three channels and fp64 go through the single-op composition; under deterministic() two runs are
    bit-identical."""
    n, h, w = 2, 24, 40
    f1, f2 = _flows(9, n, h, w, 2.0)
    for c, dtype in ((5, torch.float32), (3, torch.float64)):
        img1, img2, gt = (t.to(dtype) for t in _frames(31, n, c, h, w))
        a, b = f1.to(dtype), f2.to(dtype)
        fused_r, res_r, of_r, ob_r = _recipe_bidir(orc, img1, img2, a, b, gt)
        fused, res, of, ob = dcb.residual_conditioning_bidir(*(t.cuda() for t in (img1, img2, a, b, gt)), return_masks=True)
        assert fused.dtype == dtype and fused.shape == (n, c, h, w)
        agree = ((of.cpu().to(of_r.dtype) == of_r) & (ob.cpu().to(ob_r.dtype) == ob_r))
        assert agree.float().mean() > 0.995
        sel = agree.expand_as(fused_r)
        assert_close(fused.cpu()[sel], fused_r[sel], 1e-5, f"fused C={c} {dtype}")
        assert_close(res.cpu()[sel], res_r[sel], 1e-5, f"residual C={c} {dtype}")
    dev = [t.cuda() for t in (*_frames(32, n, 3, h, w)[:2], f1, f2, _frames(33, n, 3, h, w)[2])]
    with dcb.deterministic(True):
        r1 = dcb.residual_conditioning_bidir(*dev, return_masks=True)
        r2 = dcb.residual_conditioning_bidir(*dev, return_masks=True)
    for x, y in zip(r1, r2):
        assert torch.equal(x, y)


@pytest.mark.gpu
def test_bidir_abi_errors(dcb):
    L = dcb._lib
    lib = L.lib()
    n, c, h, w = 2, 3, 32, 48
    mk = lambda ch, dt=torch.float32: torch.rand(n, ch, h, w, device="cuda", dtype=dt)
    img1, img2, gt, f1, f2 = mk(c), mk(c), mk(c), mk(2), mk(2)
    fused, res = torch.empty_like(img1), torch.empty_like(img1)
    need = lib.dcb_residual_workspace_bytes(n, c, h, w)
    ws = torch.zeros(need + 256, dtype=torch.uint8, device="cuda")
    st = L.stream_ptr(img1.device)

    def call(i1, i2, a, b, g, fo, ro, ptr=ws.data_ptr(), nbytes=need):
        return lib.dcb_residual_bidir(L.desc(i1), L.desc(i2), L.desc(a), L.desc(b), L.desc(g), L.desc(fo), L.desc(ro), None, None,
                                      ptr, nbytes, 0, st)

    assert call(img1, img2, f1, f2, gt, fused, res) == 0
    torch.cuda.synchronize()
    assert call(img1, img2[:, :2], f1, f2, gt, fused, res) == L.E_SHAPE
    assert call(img1, img2.bfloat16(), f1, f2, gt, fused, res) == L.E_DTYPE
    four = mk(4)
    assert call(four, four, f1, f2, four, torch.empty_like(four), torch.empty_like(four)) == L.E_LIMIT
    assert call(img1, img2, f1, f2, gt, fused, res, nbytes=need - 1) == L.E_WORKSPACE
    assert call(img1, img2, f1, f2, gt, fused, res, ptr=None, nbytes=0) == L.E_WORKSPACE
    assert "workspace" in lib.dcb_last_error().decode()


@pytest.mark.gpu
def test_bidir_cuda_graph_replay(dcb):
    """One capture of the call, replayed after the inputs change: the same result as an eager call on the new inputs."""
    n, c, h, w = 2, 3, 96, 120
    img1, img2, gt = (t.cuda() for t in _frames(41, n, c, h, w))
    f1, f2 = (t.cuda() for t in _flows(11, n, h, w, 2.0))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        dcb.residual_conditioning_bidir(img1, img2, f1, f2, gt)            # warm-up: workspace allocation on this stream
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            out = dcb.residual_conditioning_bidir(img1, img2, f1, f2, gt, return_masks=True)
    torch.cuda.synchronize()
    n1, n2, ng = (t.cuda() for t in _frames(42, n, c, h, w))
    m1, m2 = (t.cuda() for t in _flows(12, n, h, w, 2.0))
    for dst, src in ((img1, n1), (img2, n2), (gt, ng), (f1, m1), (f2, m2)):
        dst.copy_(src)
    graph.replay()
    torch.cuda.synchronize()
    ref = dcb.residual_conditioning_bidir(n1, n2, m1, m2, ng, return_masks=True)
    assert torch.equal(out[2], ref[2]) and torch.equal(out[3], ref[3])
    assert_close(out[0], ref[0], 2e-6, "graph replay fused")
    assert_close(out[1], ref[1], 2e-6, "graph replay residual")
