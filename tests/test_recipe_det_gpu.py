"""The deterministic conditioning recipes (dcb_residual_fused / dcb_residual_bidir with DCB_FLAG_DETERMINISTIC, csrc/recipe.cu):
in fp32 bit for bit the composition of the deterministic single ops (residual_utils._composed / _composed_bidir under
deterministic()), masks included; 11 launches per frame group; reproducibility across runs, batch position, frame grouping and
CUDA-graph replay; the bench's deterministic residual hash; the raw ABI's workspace query and argument checks on the CPU."""
import ctypes
import importlib

import pytest
import torch
import torch.nn.functional as F

KINDS = ("dataset", "wrapper", "bidir")
SMALL = (2, 16, 24)          # 384 pixels: the non-deterministic path sends these to the cluster kernel
RAGGED = (3, 37, 53)         # H, W no multiples of 32
BATCH5 = (5, 45, 67)


@pytest.fixture(scope="module")
def dcb():
    import diffcodec_b200
    return diffcodec_b200


@pytest.fixture(scope="module")
def ru(dcb):
    return importlib.import_module(dcb.__name__ + ".residual_utils")


def _inputs(seed, n, c, h, w, flows="random"):
    """image1, image2, flow1, flow2, gt on the GPU (fp32)."""
    g = torch.Generator().manual_seed(seed)
    image1, image2, gt = (torch.rand(n, c, h, w, generator=g) for _ in range(3))
    if flows == "collide":                                        # every source of both flows lands near one pixel
        ys, xs = torch.meshgrid(torch.arange(h, dtype=torch.float32), torch.arange(w, dtype=torch.float32), indexing="ij")
        f1 = torch.stack([w / 3 - xs, h / 2 - ys]).expand(n, 2, h, w) + 0.3 * torch.rand(n, 2, h, w, generator=g)
        f2 = torch.stack([w / 2 - xs, h / 3 - ys]).expand(n, 2, h, w) + 0.3 * torch.rand(n, 2, h, w, generator=g)
    else:
        f1 = F.avg_pool2d(torch.randn(n, 2, h, w, generator=g), 5, stride=1, padding=2) * 12
        f2 = -f1 + 0.4 * torch.randn(n, 2, h, w, generator=g)
    f1, f2 = f1.contiguous(), f2.contiguous()
    for fl in (f1, f2):                                           # non-finite and out-of-frame sources
        fl[0, 0, 1, 2] = float("nan"); fl[0, 1, 2, 1] = float("inf"); fl[-1, 0, 3, 3] = float("-inf")
        fl[-1, 1, h - 1, 0] = 1e3; fl[0, 0, 0, w - 1] = -2.5 * w; fl[-1, 1, 0, 0] = float("nan")
    return tuple(t.cuda() for t in (image1, image2, f1, f2, gt))


def _library(dcb, kind, image1, image2, flow1, flow2, gt):
    if kind == "bidir":
        return dcb.residual_conditioning_bidir(image1, image2, flow1, flow2, gt, return_masks=True)
    return dcb.residual_conditioning(image1, flow1, flow2, gt, kind, return_masks=True)


def _composition(ru, kind, image1, image2, flow1, flow2, gt):
    if kind == "bidir":
        return ru._composed_bidir(image1, image2, flow1, flow2, gt)
    return ru._composed(image1, flow1, flow2, gt, kind)


NAMES = ("fused", "residual", "occ_fwd", "occ_bwd")


def _check_equal(got, ref, what):
    for name, a, b in zip(NAMES, got, ref):
        assert a.dtype == b.dtype and a.shape == b.shape, (what, name)
        assert torch.equal(a, b), f"{what}: {name} differs from the composition"


@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 2, 3])
@pytest.mark.parametrize("shape,flows", [(SMALL, "random"), (RAGGED, "random"), (BATCH5, "random"), (RAGGED, "collide")])
@pytest.mark.parametrize("kind", KINDS)
def test_equals_deterministic_composition(dcb, ru, kind, shape, flows, c):
    n, h, w = shape
    ins = _inputs(11 + c, n, c, h, w, flows)
    with dcb.deterministic():
        before = dcb.launch_count()
        got = _library(dcb, kind, *ins)
        launches = dcb.launch_count() - before
        ref = _composition(ru, kind, *ins)
    assert launches == 11, launches                               # one frame group: emit, 8 sort passes, reduce, fuse
    _check_equal(got, ref, f"{kind} {shape} {flows} C={c}")
    if flows == "random":                                          # both mask values occur
        assert 0 < got[2].sum() < got[2].numel() and 0 < got[3].sum() < got[3].numel()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_1080p_frame_equals_composition(dcb, ru, kind):
    ins = _inputs(21, 1, 3, 1080, 1920)
    with dcb.deterministic():
        before = dcb.launch_count()
        got = _library(dcb, kind, *ins)
        launches = dcb.launch_count() - before
        ref = _composition(ru, kind, *ins)
    assert launches == 11
    _check_equal(got, ref, f"{kind} 1080p")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_strided_and_expanded_inputs(dcb, ru, kind):
    n, c, h, w = 4, 3, 41, 70
    image1, image2, flow1, flow2, gt = _inputs(31, n, c, h, w)
    gt = torch.cat([gt, gt[:, :1]], dim=1)[:, 1:]                 # channel-sliced view
    image1 = image1.contiguous(memory_format=torch.channels_last)
    flow1 = torch.cat([flow1, flow1], dim=3)[..., ::2]            # strided along W
    if kind == "bidir":
        image2 = image2[:1].expand(n, c, h, w)                    # one I-frame serving every inter frame (stride 0)
    with dcb.deterministic():
        got = _library(dcb, kind, image1, image2, flow1, flow2, gt)
        ref = _composition(ru, kind, image1, image2, flow1, flow2, gt)
        dense = _library(dcb, kind, *(t.contiguous() for t in (image1, image2, flow1, flow2, gt)))
    _check_equal(got, ref, f"{kind} strided")
    _check_equal(got, dense, f"{kind} strided vs contiguous")


@pytest.mark.gpu
def test_flows_cast_as_the_composition_casts_them(dcb, ru):
    image1, image2, flow1, flow2, gt = _inputs(32, 2, 3, 33, 47)
    f1, f2 = flow1.double(), flow2.to(torch.bfloat16)
    with dcb.deterministic():
        got = dcb.residual_conditioning(image1, f1, f2, gt, "wrapper", return_masks=True)
        ref = ru._composed(image1, f1.float(), f2.float(), gt, "wrapper")
        gotb = dcb.residual_conditioning_bidir(image1, image2, f1, f2, gt.double(), return_masks=True)
        refb = ru._composed_bidir(image1, image2, f1.float(), f2.float(), gt)
    _check_equal(got, ref, "fp64 / bf16 flows")
    _check_equal(gotb, refb, "bidir, fp64 gt")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_reproducible_runs_position_grouping(dcb, ru, kind, monkeypatch):
    n, c, h, w = 5, 3, 64, 96
    ins = _inputs(41, n, c, h, w)
    with dcb.deterministic():
        runs = [_library(dcb, kind, *ins) for _ in range(3)]
        k = 3
        alone = _library(dcb, kind, *(t[k:k + 1] for t in ins))
        need = dcb._lib.lib().dcb_residual_det_workspace_bytes
        monkeypatch.setattr(ru, "DET_GROUP_BYTES", need(1, c, h, w))              # one frame per group
        before = dcb.launch_count()
        ones = _library(dcb, kind, *ins)
        assert dcb.launch_count() - before == 11 * n
        monkeypatch.setattr(ru, "DET_GROUP_BYTES", need(2, c, h, w))              # groups of two, and a last of one
        before = dcb.launch_count()
        twos = _library(dcb, kind, *ins)
        assert dcb.launch_count() - before == 11 * 3
    for r in runs[1:] + [ones, twos]:
        _check_equal(r, runs[0], f"{kind}: run / grouping")
    for a, b in zip(runs[0], alone):
        assert torch.equal(a[k:k + 1], b)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_raw_call_replays_in_a_cuda_graph(dcb, kind):
    R = dcb._lib
    lib = R.lib()
    n, c, h, w = 3, 3, 37, 53
    image1, image2, flow1, flow2, gt = _inputs(51, n, c, h, w)
    outs = [torch.empty(n, c, h, w, device="cuda"), torch.empty(n, c, h, w, device="cuda"),
            torch.empty(n, 1, h, w, device="cuda"), torch.empty(n, 1, h, w, device="cuda")]
    need = lib.dcb_residual_det_workspace_bytes(n, c, h, w)
    ws = torch.full((need,), 0xFF, dtype=torch.uint8, device="cuda")            # plain scratch: any contents
    d = R.desc

    def call(stream):
        o = [d(t) for t in outs]
        if kind == "bidir":
            return lib.dcb_residual_bidir(d(image1), d(image2), d(flow1), d(flow2), d(gt), *o, ws.data_ptr(), need,
                                          R.FLAG_DETERMINISTIC, stream)
        return lib.dcb_residual_fused(d(image1), d(flow1), d(flow2), d(gt), *o, ws.data_ptr(), need,
                                      R.RECIPE_DATASET if kind == "dataset" else R.RECIPE_WRAPPER, R.FLAG_DETERMINISTIC, stream)

    assert call(R.stream_ptr(ws.device)) == 0
    eager = [t.clone() for t in outs]
    for t in outs:
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
    for a, b in zip(outs, eager):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_bench_hash_of_two_gops_equals_the_composition(dcb, ru):
    """bench.py's deterministic residual hash (C5), for the first two GOPs of the sweep: one call against the composition."""
    H, W = 1080, 1920
    dev = torch.device("cuda")
    total = {"call": 0, "composition": 0}
    for u in dcb.enumerate_gops()[:2]:
        gen = torch.Generator(device=dev).manual_seed(u.seed())
        k = u.inter_frames
        img, gt = torch.empty(k, 3, H, W, device=dev), torch.empty(k, 3, H, W, device=dev)
        low1, low2 = torch.empty(k, 2, H // 32, W // 32, device=dev), torch.empty(k, 2, H // 32, W // 32, device=dev)
        img.uniform_(generator=gen); gt.uniform_(generator=gen); low1.normal_(generator=gen); low2.normal_(generator=gen)
        f1 = F.interpolate(low1, size=(H, W), mode="bicubic", align_corners=False) * 8.0
        f2 = -f1 + 0.5 * F.interpolate(low2, size=(H, W), mode="bicubic", align_corners=False)
        with dcb.deterministic():
            _, res = dcb.residual_conditioning(img, f1, f2, gt, "dataset")
            _, ref, _, _ = ru._composed(img, f1, f2, gt, "dataset")
        assert torch.equal(res, ref)
        total["call"] += int(res.contiguous().view(torch.int32).to(torch.int64).sum())
        total["composition"] += int(ref.contiguous().view(torch.int32).to(torch.int64).sum())
    assert total["call"] == total["composition"]


@pytest.mark.gpu
def test_bf16_fp64_and_wide_keep_the_composition(dcb, ru):
    image1, image2, flow1, flow2, gt = _inputs(61, 2, 3, 24, 40)
    with dcb.deterministic():
        for dt in (torch.bfloat16, torch.float64):
            a = [t.to(dt) for t in (image1, flow1, flow2, gt)]
            got = dcb.residual_conditioning(*a, "wrapper", return_masks=True)
            ref = ru._composed(*a, "wrapper")
            _check_equal(got, ref, f"{dt}")
        wide = [torch.cat([t, t], dim=1) for t in (image1, image2, gt)]
        got = dcb.residual_conditioning_bidir(wide[0], wide[1], flow1, flow2, wide[2], return_masks=True)
        _check_equal(got, ru._composed_bidir(wide[0], wide[1], flow1, flow2, wide[2]), "C = 6")


# ---------------------------------------------------------------------------------------------
# CPU: the workspace query and the argument checks read descriptors only (fake device addresses, nothing is launched)
# ---------------------------------------------------------------------------------------------
class _Fakes:
    def __init__(self):
        self.keep, self.addr = [], 1 << 32

    def __call__(self, n, c, h, w, dtype=None, offset=0):
        from diffcodec_b200 import _lib
        b = ctypes.create_string_buffer(_lib._DESC_STRUCT.pack(self.addr + offset, _lib.DCB_F32 if dtype is None else dtype, 0,
                                                               n, c, h, w, c * h * w, h * w, w, 1))
        self.addr += 1 << 38
        self.keep.append(b)
        return ctypes.addressof(b)


def _calls(n, c, h, w, dtype=None):
    from diffcodec_b200 import _lib
    lib = _lib.lib()
    d = _Fakes()
    img, img2, f1, f2, gt = d(n, c, h, w, dtype), d(n, c, h, w, dtype), d(n, 2, h, w, dtype), d(n, 2, h, w, dtype), d(n, c, h, w, dtype)
    outs = (d(n, c, h, w, dtype), d(n, c, h, w, dtype), d(n, 1, h, w, dtype), d(n, 1, h, w, dtype))

    def fused(ws, nbytes, flags):
        return lib.dcb_residual_fused(img, f1, f2, gt, *outs, ws, nbytes, _lib.RECIPE_DATASET, flags, None)

    def bidir(ws, nbytes, flags):
        return lib.dcb_residual_bidir(img, img2, f1, f2, gt, *outs, ws, nbytes, flags, None)
    return (fused, bidir), d


def test_det_workspace_query_and_argument_checks_cpu():
    from diffcodec_b200 import _lib
    lib = _lib.lib()
    n, c, h, w = 3, 3, 1080, 1920
    need = lib.dcb_residual_det_workspace_bytes(n, c, h, w)
    keys = 8 * n * h * w
    cells = n * h * w * (48 + 2 * 16)                                  # mask and normaliser planes + one feature quad per flow
    assert need >= 2 * 8 * keys + cells                                # keys and sorted keys on top of the cells
    assert lib.dcb_residual_det_workspace_bytes(n, 1, h, w) == lib.dcb_residual_det_workspace_bytes(n, 3, h, w)
    assert lib.dcb_residual_det_workspace_bytes(2 * n, c, h, w) > need
    for bad in ((-1, c, h, w), (n, -1, h, w), (n, c, -1, w), (n, c, h, -1)):
        assert lib.dcb_residual_det_workspace_bytes(*bad) == 0
    DET, CLEAN = _lib.FLAG_DETERMINISTIC, _lib.FLAG_WS_CLEAN
    big = 1 << 40
    (fused, bidir), _ = _calls(n, c, h, w)
    for call in (fused, bidir):
        assert call(big, big, DET | CLEAN) == _lib.E_MODE
        assert call(big, need - 1, DET) == _lib.E_WORKSPACE
        assert call(big + 16, big, DET) == _lib.E_WORKSPACE
        assert call(None, 0, DET) == _lib.E_WORKSPACE
    assert bidir(big, big, DET | 16) == _lib.E_MODE                   # dcb_residual_bidir still refuses unknown bits
    (fused16, bidir16), _ = _calls(n, c, h, w, _lib.DCB_BF16)
    assert fused16(big, big, DET) == _lib.E_DTYPE and bidir16(big, big, DET) == _lib.E_DTYPE
    # 8 keys per pixel: 8 * 16384 * 16384 = 2^31 keys is one too many; one row less fits (and wants its workspace)
    (fh, bh), _ = _calls(1, 3, 16384, 16384)
    assert fh(big, big, DET) == _lib.E_LIMIT and bh(big, big, DET) == _lib.E_LIMIT
    (ff, bf), _ = _calls(1, 3, 16383, 16384)
    assert ff(big, 256, DET) == _lib.E_WORKSPACE and bf(big, 256, DET) == _lib.E_WORKSPACE
    assert lib.dcb_residual_det_workspace_bytes(1, 3, 16383, 16384) > 2 * 8 * 8 * 16383 * 16384
