"""The backward kernels in the forms training runs, against the CPU oracle through torch autograd.

A training step rarely wants every gradient with NCHW inputs and a contiguous upstream gradient: the flow is often frozen,
features arrive channels_last, and a loss reduced to a scalar hands the kernel an expanded (stride-0) gradient. Each of
these selects its own kernel or kernel form:

  * splat backward, packed path (C <= 3, normalised modes, fp32/bf16/fp16, csrc/splat_bwd.cu): the compile-time "flat"
    source pass (all gradients, NCHW) and the run-time form (any subset, any strides), frame groups, the (1 - mask) factor;
  * splat backward, generic path: channel slices (cs > 1 / ct > 1), cs = 1, sum mode, fp64, and the 64-bit gradOut
    offsets of k_bwd_source<..., long long>;
  * backward warp (csrc/backwarp.cu): fp64, bf16 through the fp32 workspace and the cast kernel, gradient subsets, the
    residual / gt gradients, huge and non-finite flows, an image view whose offsets need 64 bits;
  * fusion backward (csrc/fuse.cu): gradient subsets, confidences of exactly 0, double holes.

Every test compares the CUDA result with the oracle (oracle/oracle.py) run through autograd with the same requires_grad
pattern. Tolerances (DESIGN.md section 2): 1e-5 relative in fp32, widened by the fp64 truth where the fp32 reference is
ill-conditioned (tests/util.assert_close); 1e-12 in fp64; 1e-2 in bf16/fp16 against the fp32 oracle on the up-cast inputs.
The 64-bit-offset tests compare two GPU runs that differ only in the index type, bit for bit."""
import importlib
import itertools
import zlib

import pytest
import torch

from tests.util import assert_close, make_inputs

pytestmark = pytest.mark.gpu

NAMES = ("in", "flow", "metric")


@pytest.fixture(scope="module")
def dcb():
    import diffcodec_b200
    return diffcodec_b200


@pytest.fixture(scope="module")
def impl(dcb):
    return importlib.import_module(dcb.__name__ + ".softsplat")      # the submodule (the package re-exports the function)


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    oracle.lib()
    return oracle


@pytest.fixture
def option(dcb):
    """set(name, value) for library options; each option touched is back at its default afterwards, and the workspaces
    sized under it are released."""
    L = dcb._lib
    defaults = {"bwd_flat": 1, "bwd_group_bytes": 0, "fwd_path": 0}
    touched = set()

    def set_(name, value):
        touched.add(name)
        L.set_option(name, value)
        L.release_workspaces()
    try:
        yield set_
    finally:
        for name in touched:
            L.set_option(name, defaults[name])
        L.release_workspaces()


def _seed(*key):
    return zlib.crc32(repr(key).encode()) % 1000          # stable across processes (str hash is salted)


def _has_metric(mode):
    return mode.split("-")[0] in ("linear", "soft")


def _subsets(mode):
    names = NAMES if _has_metric(mode) else NAMES[:2]
    return [s for r in range(1, len(names) + 1) for s in itertools.combinations(names, r)]


def _splat_inputs(mode, n, c, h, w, flow_scale=2.5, seed=None):
    tin, flow, metric, gout = make_inputs(_seed(mode, n, c, h, w) if seed is None else seed, n, c, h, w, flow_scale=flow_scale)
    if mode.startswith("linear"):
        metric = metric.abs() + 0.1          # keep the normaliser away from cancellation (the tolerance is relative)
    return tin, flow, metric if _has_metric(mode) else None, gout


def run_splat(fn, tin, flow, metric, gout, want, device="cpu", views=None):
    """fn(in, flow, metric) -> out with autograd. Leaves require grad as `want` says; `views` maps a name to a function of
    its leaf that gives the tensor the op sees (a layout), so the gradient still lands on the NCHW leaf.
    Returns (out, {name: grad or None})."""
    leaves = {}
    for k, t in zip(NAMES, (tin, flow, metric)):
        if t is None:
            leaves[k] = None
            continue
        leaves[k] = t.detach().to(device).clone().requires_grad_(k in want)
    args = [None if leaves[k] is None else (views[k](leaves[k]) if views and k in views else leaves[k]) for k in NAMES]
    out = fn(*args)
    out.backward(gout.to(device=device, dtype=out.dtype))
    return out.detach(), {k: None if leaves[k] is None else leaves[k].grad for k in NAMES}


def check_splat(got, ref, want, rel, what, truth=None):
    assert_close(got[0], ref[0], rel, f"{what} out", truth=None if truth is None else truth[0])
    for k in NAMES:
        if k in want:
            assert got[1][k] is not None, f"{what}: grad {k} missing"
            assert_close(got[1][k], ref[1][k], rel, f"{what} grad {k}", truth=None if truth is None else truth[1][k])
        else:
            assert got[1][k] is None, f"{what}: grad {k} was not asked for"


def _cuda_splat(dcb, mode):
    return lambda i, f, m: dcb.softsplat(i, f, m, mode)


def _orc_splat(orc, mode):
    return lambda i, f, m: orc.softsplat(i, f, m, mode)


def _oracle_pair(orc, mode, tin, flow, metric, gout, want):
    ref = run_splat(_orc_splat(orc, mode), tin, flow, metric, gout, want)
    truth = run_splat(_orc_splat(orc, mode), tin.double(), flow.double(), None if metric is None else metric.double(),
                      gout.double(), want)
    return ref, truth


# ---------------------------------------------------------------------------------------------------------------------
# A. Splat backward: gradient subsets x kernel form x dtype
# ---------------------------------------------------------------------------------------------------------------------
SUBSET_MODES = ["sum", "avg", "linear", "soft", "soft-clipeps", "linear-zeroeps"]
# C = 1, 2, 3: the packed path (flat form for all gradients, run-time form for a subset; 'sum' takes the generic path with
# no target pass). C = 19 / 65 on a few pixels: the generic path with channel slices in both passes (cs = 16 / 32,
# ct = 2 / 8), channel counts not divisible by the slice count.
SUBSET_SHAPES = [(2, 1, 17, 40), (3, 2, 16, 16), (2, 3, 24, 33), (2, 19, 8, 8), (1, 65, 6, 10)]
# the default seed of this case lets a target pixel receive nothing but a ~1e-16 bilinear weight: with zeroeps its
# normaliser is that weight, the gradients there reach 1e15 x their median and a max-scaled tolerance checks nothing else
SUBSET_SEEDS = {("linear-zeroeps", (1, 65, 6, 10)): 1000}


@pytest.mark.parametrize("mode", SUBSET_MODES)
@pytest.mark.parametrize("shape", SUBSET_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_splat_gradient_subsets(dcb, orc, mode, shape):
    """Every non-empty subset of {in, flow, metric} the mode allows: the wanted gradients match the oracle run with the same
    requires_grad pattern and the all-gradients CUDA run; the others are None."""
    tin, flow, metric, gout = _splat_inputs(mode, *shape, seed=SUBSET_SEEDS.get((mode, shape)))
    full_want = NAMES if _has_metric(mode) else NAMES[:2]
    full = run_splat(_cuda_splat(dcb, mode), tin, flow, metric, gout, full_want, "cuda")
    for want in _subsets(mode):
        ref, truth = _oracle_pair(orc, mode, tin, flow, metric, gout, want)
        for k in want:                                         # the max-scaled tolerance must still see ordinary elements
            a = truth[1][k].abs()
            assert a.max() <= 1e4 * a.median(), f"{mode} {shape}: grad {k} is ill-conditioned; pick another seed"
        got = run_splat(_cuda_splat(dcb, mode), tin, flow, metric, gout, want, "cuda")
        check_splat(got, ref, want, 1e-5, f"{mode} {shape} {want}", truth)
        for k in want:
            assert_close(got[1][k], full[1][k], 1e-6, f"{mode} {shape} {want}: grad {k} vs the all-gradients run")


@pytest.mark.parametrize("mode", ["avg", "linear", "soft", "soft-clipeps"])
@pytest.mark.parametrize("c", [1, 2, 3])
def test_packed_flat_and_runtime_forms_agree(dcb, orc, option, mode, c):
    """All gradients on NCHW frames take the compile-time form k_bwd_source4<T, TF, C, MODE>; bwd_flat = 0 sends the same
    call through the run-time form k_bwd_source4<T, TF, 0, 0>. Both match the oracle and each other."""
    tin, flow, metric, gout = _splat_inputs(mode, 2, c, 24, 40)
    want = NAMES if _has_metric(mode) else NAMES[:2]
    ref, truth = _oracle_pair(orc, mode, tin, flow, metric, gout, want)
    flat = run_splat(_cuda_splat(dcb, mode), tin, flow, metric, gout, want, "cuda")
    option("bwd_flat", 0)
    runtime = run_splat(_cuda_splat(dcb, mode), tin, flow, metric, gout, want, "cuda")
    check_splat(flat, ref, want, 1e-5, f"flat C={c} {mode}", truth)
    check_splat(runtime, ref, want, 1e-5, f"run-time C={c} {mode}", truth)
    for k in want:
        assert_close(runtime[1][k], flat[1][k], 1e-6, f"C={c} {mode}: run-time vs flat grad {k}")


@pytest.mark.parametrize("want", [("in", "flow", "metric"), ("flow", "metric"), ("in",)], ids="+".join)
def test_generic_path_one_slice(dcb, orc, want):
    """303,104 pixels (148 x 2048) with C = 4: the generic backward runs one channel slice per pixel (cs = ct = 1) and its L2
    prefetch."""
    n, c, h, w = 1, 4, 512, 592
    assert n * h * w >= 148 * 2048
    tin, flow, metric, gout = _splat_inputs("soft", n, c, h, w, flow_scale=3.0)
    ref, truth = _oracle_pair(orc, "soft", tin, flow, metric, gout, want)
    got = run_splat(_cuda_splat(dcb, "soft"), tin, flow, metric, gout, want, "cuda")
    check_splat(got, ref, want, 1e-5, f"cs=1 {want}", truth)


@pytest.mark.parametrize("mode", ["sum", "avg", "soft", "linear-zeroeps"])
def test_fp64_gradient_subsets(dcb, orc, mode):
    """fp64 always takes the generic path (k_bwd_target<double>, k_bwd_source<double, double, int>): every subset at 1e-12."""
    tin, flow, metric, gout = (None if t is None else t.double() for t in _splat_inputs(mode, 2, 3, 17, 19, flow_scale=3.0))
    for want in _subsets(mode):
        ref = run_splat(_orc_splat(orc, mode), tin, flow, metric, gout, want)
        got = run_splat(_cuda_splat(dcb, mode), tin, flow, metric, gout, want, "cuda")
        check_splat(got, ref, want, 1e-12, f"fp64 {mode} {want}")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=str)
@pytest.mark.parametrize("flow_dtype", ["f32", "same"])
@pytest.mark.parametrize("shape", [(2, 3, 24, 40), (2, 19, 8, 8)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("mode", ["avg", "soft"])
def test_16bit_gradient_subsets(dcb, orc, dtype, flow_dtype, shape, mode):
    """bf16 / fp16 data (an fp32 flow or one of the data's dtype): the packed path at C = 3 (flat and run-time forms), the
    generic path at C = 19. Within 1e-2 of the fp32 oracle on the up-cast inputs."""
    # flows below ~half a pixel keep every normaliser O(1): with a tiny normaliser the saved 16-bit output is amplified by
    # 1/D in the gradients, for the reference as for us
    tin, flow, metric, gout = _splat_inputs(mode, *shape, flow_scale=0.4)
    cast = lambda t: None if t is None else t.to(dtype)
    tin, metric, gout = cast(tin), cast(metric), cast(gout)
    if flow_dtype == "same":
        flow = flow.to(dtype)
    for want in (_subsets(mode)[-1], ("flow",) + (("metric",) if metric is not None else ()), ("in",)):
        ref = run_splat(_orc_splat(orc, mode), tin.float(), flow.float(), None if metric is None else metric.float(),
                        gout.float(), want)
        got = run_splat(_cuda_splat(dcb, mode), tin, flow, metric, gout, want, "cuda")
        assert got[0].dtype == dtype
        if "flow" in want:
            assert got[1]["flow"].dtype == flow.dtype
        check_splat((got[0].float(), {k: None if v is None else v.float() for k, v in got[1].items()}), ref, want, 1e-2,
                    f"{dtype} flow={flow_dtype} {mode} {want}")


@pytest.mark.parametrize("want", [("flow", "metric"), ("in", "metric"), ("in", "flow", "metric")], ids="+".join)
def test_frame_groups_with_subsets(dcb, orc, option, want):
    """Five frames in groups of two (the last one short): target and source passes alternate on one slot of packed cells."""
    n, c, h, w = 5, 3, 20, 36
    option("bwd_group_bytes", 2 * h * w * 16)
    tin, flow, metric, gout = _splat_inputs("soft", n, c, h, w, flow_scale=3.0)
    ref, truth = _oracle_pair(orc, "soft", tin, flow, metric, gout, want)
    L = dcb._lib
    assert L.lib().dcb_splat_bwd_workspace_bytes(n, c, h, w, L._DTYPES[torch.float32], L.MODE_SOFT, 0) == 2 * h * w * 16
    got = run_splat(_cuda_splat(dcb, "soft"), tin, flow, metric, gout, want, "cuda")
    check_splat(got, ref, want, 1e-5, f"frame groups {want}", truth)


def _channels_last(t):
    return t.contiguous(memory_format=torch.channels_last)


def _flow_slice(f):
    return torch.cat([f[:, :1] * 0 + 5.0, f, f[:, :1] * 0 - 7.0], 1)[:, 1:3]          # flow[:, 1:3] of a 4-channel tensor


def _metric_slice(m):
    return torch.cat([m * 0 + 3.0, m, m * 0 - 3.0], 1)[:, 1:2]


def _row_padded(t):
    return torch.cat([t, t[..., :5] * 0 + 9.0], 3)[..., :t.shape[3]]         # rows 5 elements longer than W: sH = W + 5


# flow[:, 1:3] and a metric channel slice keep NCHW strides inside a frame (only sN changes); a channels_last flow
# (sC = 1, sW = 2) and row-padded flow / metric (sH = W + 5) do not, and force the run-time form even with every gradient
LAYOUTS = {"in_channels_last": {"in": _channels_last}, "flow_slice": {"flow": _flow_slice},
           "metric_slice": {"metric": _metric_slice}, "flow_channels_last": {"flow": _channels_last},
           "flow_metric_row_padded": {"flow": _row_padded, "metric": _row_padded},
           "all": {"in": _channels_last, "flow": _flow_slice, "metric": _metric_slice}}


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("c", [3, 19])
@pytest.mark.parametrize("want", [("in", "flow", "metric"), ("flow",)], ids="+".join)
def test_input_layouts(dcb, orc, layout, c, want):
    """channels_last features, a sliced flow and a sliced metric, through the packed (C = 3) and generic (C = 19) backward:
    the oracle's values, and those of the contiguous call."""
    tin, flow, metric, gout = _splat_inputs("soft", 2, c, 20, 28)
    ref, truth = _oracle_pair(orc, "soft", tin, flow, metric, gout, want)
    got = run_splat(_cuda_splat(dcb, "soft"), tin, flow, metric, gout, want, "cuda", views=LAYOUTS[layout])
    base = run_splat(_cuda_splat(dcb, "soft"), tin, flow, metric, gout, want, "cuda")
    check_splat(got, ref, want, 1e-5, f"{layout} C={c} {want}", truth)
    for k in want:
        assert_close(got[1][k], base[1][k], 1e-6, f"{layout} C={c}: grad {k} vs the contiguous call")


# ---------------------------------------------------------------------------------------------------------------------
# B. Masks and upstream-gradient layouts
# ---------------------------------------------------------------------------------------------------------------------
def _mask_case(c, seed):
    """Smooth small flows, a mask with an all-ones block (rows 6..13, cols 8..19) and scattered ones, and a block of very
    negative metric (rows 1..11, cols 20..34 of a 16 x 36 frame) where only tiny weights land: the clip of clipeps is active."""
    n, h, w = 2, 16, 36
    tin, flow, metric, gout = make_inputs(seed, n, c, h, w, flow_scale=0.6, smooth=True)
    g = torch.Generator().manual_seed(seed + 1)
    mask = (torch.rand(n, 1, h, w, generator=g) > 0.8).float()
    mask[:, :, 6:14, 8:20] = 1.0
    metric[:, :, 1:12, 20:35] = -30.0
    return tin, flow, metric, gout, mask


def _inside_block(flow, y0, y1, x0, x1):
    """Source pixels whose four bilinear corners all land inside rows y0..y1-1, cols x0..x1-1 (with a margin)."""
    n, _, h, w = flow.shape
    ys, xs = torch.meshgrid(torch.arange(h, dtype=torch.float64), torch.arange(w, dtype=torch.float64), indexing="ij")
    tx, ty = xs + flow[:, 0].double(), ys + flow[:, 1].double()
    e = 1e-3
    return (tx >= x0 + e) & (tx <= x1 - 1 - e) & (ty >= y0 + e) & (ty <= y1 - 1 - e)


@pytest.mark.parametrize("mode", ["soft", "soft-clipeps"])
@pytest.mark.parametrize("c", [1, 2, 3, 19])
def test_mask_factor(dcb, orc, impl, mode, c):
    """_splat_normalised(..., mask=m), as FeatureWarperSoftsplat calls it: the (1 - mask) factor of the target pass
    (k_bwd_target4 at C <= 3, k_bwd_target at C = 19) against the oracle's feature_warper, in full and in the block where
    the clip is active; exactly 0 output inside the all-ones block of the mask, and exactly 0 gradIn at every source pixel
    whose four corners land inside it."""
    tin, flow, metric, gout, mask = _mask_case(c, _seed("mask", mode, c))
    eps = dcb._lib.EPS_CLIP if mode == "soft-clipeps" else dcb._lib.EPS_ADD
    mc = mask.cuda()

    def ref_fn(i, f, m):
        if mode == "soft":
            return orc.feature_warper(i, f, m, mask)[0]
        return orc.softsplat(i, f, m, mode) * (1 - mask)

    cuda_fn = lambda i, f, m: impl._splat_normalised(i, f, m, dcb._lib.MODE_SOFT, eps, mask=mc)
    want = NAMES
    ref = run_splat(ref_fn, tin, flow, metric, gout, want)
    truth = run_splat(lambda i, f, m: (orc.feature_warper(i, f, m, mask.double())[0] if mode == "soft"
                                       else orc.softsplat(i, f, m, mode) * (1 - mask.double())),
                      tin.double(), flow.double(), metric.double(), gout.double(), want)
    got = run_splat(cuda_fn, tin, flow, metric, gout, want, "cuda")
    check_splat(got, ref, want, 1e-5, f"mask {mode} C={c}", truth)
    # the very-negative-metric block on its own scale (its values are ~1e-6 of the rest)
    blk = (slice(None), slice(None), slice(3, 10), slice(23, 32))
    for k, a, r, t in (("out", got[0], ref[0], truth[0]), ("gin", got[1]["in"], ref[1]["in"], truth[1]["in"]),
                       ("gmetric", got[1]["metric"], ref[1]["metric"], truth[1]["metric"])):
        assert_close(a[blk], r[blk], 1e-5, f"mask {mode} C={c} {k} in the low-metric block", truth=t[blk])
    if mode == "soft-clipeps":
        norm = orc.softsplat(metric.exp(), flow, None, "sum")
        assert ((norm[blk] > 0) & (norm[blk] < 1e-7)).any(), "the clip must be active somewhere in the block"
    out = got[0].cpu()
    assert (out[:, :, 6:14, 8:20] == 0).all(), "output inside the all-ones mask block must be exactly 0"
    inside = _inside_block(flow, 6, 14, 8, 20)
    assert inside.sum() >= 20
    gin = got[1]["in"].cpu()
    assert (gin.permute(1, 0, 2, 3)[:, inside] == 0).all(), "gradIn of sources landing in the all-ones block must be exactly 0"


def _upstream_grad(kind, shape):
    """An upstream gradient on the device that is not NCHW-contiguous (built there: copying a non-dense view to the device
    would give a contiguous tensor)."""
    n, c, h, w = shape
    if kind == "sum":                                            # what out.sum() hands back: ones, stride 0
        return torch.ones((), device="cuda").expand(shape)
    if kind == "mean":
        return torch.full((), 1.0 / (n * c * h * w), device="cuda").expand(shape)
    base = torch.randn(shape, generator=torch.Generator().manual_seed(_seed("layouts", kind, shape))).cuda()
    if kind == "channels_last":
        return base.contiguous(memory_format=torch.channels_last)
    if kind == "transposed":                                     # permute(0, 1, 3, 2) of a W x H tensor
        return base.transpose(2, 3).contiguous().permute(0, 1, 3, 2)
    assert kind == "channel_slice"
    return torch.cat([base[:, :1], base, base[:, :1]], 1)[:, 1:1 + c]


UPSTREAM = ["sum", "mean", "channels_last", "transposed", "channel_slice"]


def _backward_with(out, leaves, g):
    """Gradients of `out` for the upstream gradient `g` as given (its strides reach the op: checked by a hook)."""
    seen = []
    h = out.register_hook(lambda t: seen.append(t.stride()))
    grads = torch.autograd.grad(out, leaves, g, retain_graph=True)
    h.remove()
    assert seen and seen[0] == g.stride(), (seen, g.stride())
    return grads


@pytest.mark.parametrize("kind", UPSTREAM)
@pytest.mark.parametrize("case", ["packed_soft_c3", "generic_soft_c19", "generic_sum_c3"])
def test_splat_upstream_gradient_layouts(dcb, orc, kind, case):
    """The packed target pass (C = 3, soft), the generic target + source passes (C = 19, soft) and the generic source pass
    alone ('sum', C = 3) read the upstream gradient through its strides: the same gradients as for its .contiguous() copy
    (one forward, two backwards), and the oracle's."""
    mode, c = {"packed_soft_c3": ("soft", 3), "generic_soft_c19": ("soft", 19), "generic_sum_c3": ("sum", 3)}[case]
    tin, flow, metric, _ = _splat_inputs(mode, 2, c, 20, 28)
    g = _upstream_grad(kind, (2, c, 20, 28))
    assert not g.is_contiguous()
    leaves = [t.cuda().requires_grad_(True) for t in (tin, flow) + ((metric,) if metric is not None else ())]
    out = dcb.softsplat(leaves[0], leaves[1], leaves[2] if metric is not None else None, mode)
    strided = _backward_with(out, leaves, g)
    contig = torch.autograd.grad(out, leaves, g.contiguous())
    for k, a, b in zip(NAMES, strided, contig):
        assert torch.equal(a, b), f"{case} {kind}: grad {k} differs from the contiguous-gradient run"
    want = NAMES[:len(leaves)]
    gc = g.contiguous().cpu()
    ref, truth = _oracle_pair(orc, mode, tin, flow, metric, gc, want)
    for k, a in zip(NAMES, strided):
        assert_close(a, ref[1][k], 1e-5, f"{case} {kind} grad {k}", truth=truth[1][k])


@pytest.mark.parametrize("kind", UPSTREAM)
def test_backwarp_upstream_gradient_layouts(dcb, orc, kind):
    n, c, h, w = 2, 3, 20, 28
    gen = torch.Generator().manual_seed(_seed("bw layouts", kind))
    img, flow = torch.rand(n, c, h, w, generator=gen), torch.randn(n, 2, h, w, generator=gen) * 3
    g = _upstream_grad(kind, (n, c, h, w))
    leaves = [img.cuda().requires_grad_(True), flow.cuda().requires_grad_(True)]
    out = dcb.backwarp(leaves[0], leaves[1])
    strided = _backward_with(out, leaves, g)
    contig = torch.autograd.grad(out, leaves, g.contiguous())
    assert_close(strided[0], contig[0], 1e-6, f"backwarp {kind} gimage vs contiguous")      # gimage: atomic order
    assert torch.equal(strided[1], contig[1]), f"backwarp {kind} gflow vs contiguous"
    gc = g.contiguous().cpu()
    ref = _backwarp_ref(orc, img, flow, None, False, gc, None, ("image", "flow"))
    truth = _backwarp_ref(orc, img.double(), flow.double(), None, False, gc.double(), None, ("image", "flow"))
    assert_close(strided[0], ref[2]["image"], 1e-5, f"backwarp {kind} gimage", truth=truth[2]["image"])
    assert_close(strided[1], ref[2]["flow"], 1e-5, f"backwarp {kind} gflow", truth=truth[2]["flow"])


@pytest.mark.parametrize("kind", UPSTREAM)
def test_fuse_upstream_gradient_layouts(dcb, orc, kind):
    A, B, ca, cb, oa, ob = _fuse_inputs(_seed("fuse layouts", kind))
    g = _upstream_grad(kind, tuple(A.shape))
    leaves = [t.cuda().requires_grad_(True) for t in (A, B, ca, cb)]
    out = dcb.bidir_fuse(*leaves, oa.cuda(), ob.cuda())
    strided = _backward_with(out, leaves, g)
    contig = torch.autograd.grad(out, leaves, g.contiguous())
    cpu = [t.clone().requires_grad_(True) for t in (A, B, ca, cb)]
    orc.fuse(*cpu, oa, ob).backward(g.contiguous().cpu())
    for name, a, b, r in zip(FUSE_NAMES, strided, contig, cpu):
        assert torch.equal(a, b), f"fuse {kind} grad {name} vs contiguous"
        _assert_fuse_grad(name, a, r.grad, ca, cb, f"fuse {kind}")


# ---------------------------------------------------------------------------------------------------------------------
# C. Backward warp: dtype matrix and gradient subsets
# ---------------------------------------------------------------------------------------------------------------------
def _backwarp_ref(orc, img, flow, gt, align, g_warped, g_residual, want):
    """oracle.backwarp (torch's CPU grid_sample, the grid built as warp.py builds it) through autograd.
    Returns (warped, residual or None, {image, flow, gt: grad or None})."""
    leaves = {"image": img.clone().requires_grad_("image" in want), "flow": flow.clone().requires_grad_("flow" in want),
              "gt": None if gt is None else gt.clone().requires_grad_("gt" in want)}
    warped = orc.backwarp(leaves["image"], leaves["flow"], align_corners=align)
    residual = None if gt is None else leaves["gt"] - warped
    loss = 0
    if g_warped is not None:
        loss = loss + (warped * g_warped).sum()
    if g_residual is not None:
        loss = loss + (residual * g_residual).sum()
    loss.backward()
    return warped.detach(), None if residual is None else residual.detach(), {k: None if v is None else v.grad for k, v in leaves.items()}


def _backwarp_cuda(dcb, img, flow, gt, align, g_warped, g_residual, want):
    leaves = {"image": img.cuda().requires_grad_("image" in want), "flow": flow.cuda().requires_grad_("flow" in want),
              "gt": None if gt is None else gt.cuda().requires_grad_("gt" in want)}
    if gt is None:
        warped, residual = dcb.backwarp(leaves["image"], leaves["flow"], align_corners=align), None
    else:
        warped, residual = dcb.backwarp_residual(leaves["image"], leaves["flow"], leaves["gt"], align_corners=align)
    outs, grads = [], []
    if g_warped is not None:
        outs.append(warped); grads.append(g_warped.to(device="cuda", dtype=warped.dtype))
    if g_residual is not None:
        outs.append(residual); grads.append(g_residual.to(device="cuda", dtype=residual.dtype))
    torch.autograd.backward(outs, grads)
    return warped.detach(), None if residual is None else residual.detach(), {k: None if v is None else v.grad for k, v in leaves.items()}


def _warp_case(seed, n, c, h, w, scale=3.0):
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(n, c, h, w, generator=g)
    flow = torch.randn(n, 2, h, w, generator=g) * scale
    flow[:, :, :, :3] -= 0.7 * w / 4                           # taps that leave the frame on the left ...
    gt = torch.rand(n, c, h, w, generator=g)
    gw, gr = torch.randn(n, c, h, w, generator=g), torch.randn(n, c, h, w, generator=g)
    return img, flow, gt, gw, gr


def _check_warp(got, ref, want, rel, what, truth=None):
    t = (lambda i, k=None: None) if truth is None else (lambda i, k=None: truth[i] if k is None else truth[2][k])
    assert_close(got[0], ref[0], rel, f"{what} warped", truth=t(0))
    if ref[1] is not None:
        assert_close(got[1], ref[1], rel, f"{what} residual", truth=t(1))
    for k in ("image", "flow", "gt"):
        if k in want:
            assert got[2][k] is not None, f"{what}: grad {k} missing"
            assert_close(got[2][k], ref[2][k], rel, f"{what} grad {k}", truth=t(2, k))
        else:
            assert got[2][k] is None, f"{what}: grad {k} was not asked for"


WARP_SHAPES = [(2, 3, 20, 33), (2, 3, 24, 40)]        # odd W (generic forward kernel), W % 4 == 0 (paired-rows kernel)


@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("shape", WARP_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_backwarp_fp64(dcb, orc, align, shape):
    """k_backwarp_fwd<double, double> and k_backwarp_bwd<double, double>: warped, residual and the image, flow and gt
    gradients at 1e-12."""
    img, flow, gt, gw, gr = (t.double() for t in _warp_case(_seed("fp64", align, shape), *shape))
    want = ("image", "flow", "gt")
    ref = _backwarp_ref(orc, img, flow, gt, align, gw, gr, want)
    got = _backwarp_cuda(dcb, img, flow, gt, align, gw, gr, want)
    assert got[0].dtype == torch.float64 and got[2]["flow"].dtype == torch.float64
    _check_warp(got, ref, want, 1e-12, f"fp64 align={align} {shape}")


@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("shape", WARP_SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("flow_dtype", [torch.float32, torch.bfloat16], ids=str)
def test_backwarp_bf16(dcb, orc, align, shape, flow_dtype):
    """bf16 image: gimage accumulates in the fp32 workspace and is cast by k_cast_f32_bf16; gflow comes back in the flow's
    dtype. Within 1e-2 of the fp32 oracle on the up-cast inputs, for both gradients and for each alone."""
    img, flow, gt, gw, gr = _warp_case(_seed("bf16", align, shape), *shape, scale=1.5)
    ib, fb, gb = img.bfloat16(), flow.to(flow_dtype), gt.bfloat16()
    gwb = gw.bfloat16()
    for want in (("image", "flow"), ("image",), ("flow",)):
        ref = _backwarp_ref(orc, ib.float(), fb.float(), None, align, gwb.float(), None, want)
        got = _backwarp_cuda(dcb, ib, fb, None, align, gwb, None, want)
        assert got[0].dtype == torch.bfloat16
        if "image" in want:
            assert got[2]["image"].dtype == torch.bfloat16
        if "flow" in want:
            assert got[2]["flow"].dtype == flow_dtype
        _check_warp((got[0].float(), None, {k: None if v is None else v.float() for k, v in got[2].items()}), ref, want, 1e-2,
                    f"bf16 flow={flow_dtype} align={align} {shape} {want}")
    # the fused residual in bf16, with a loss on both outputs
    ref = _backwarp_ref(orc, ib.float(), fb.float(), gb.float(), align, gwb.float(), gr.bfloat16().float(), ("image", "flow", "gt"))
    got = _backwarp_cuda(dcb, ib, fb, gb, align, gwb, gr.bfloat16(), ("image", "flow", "gt"))
    _check_warp((got[0].float(), got[1].float(), {k: v.float() for k, v in got[2].items()}), ref, ("image", "flow", "gt"), 1e-2,
                f"bf16 residual flow={flow_dtype} align={align} {shape}")


@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("shape", WARP_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_backwarp_gradient_subsets_and_residual_losses(dcb, orc, align, shape):
    """fp32: gimage alone and gflow alone (equal to the both-gradients run: gflow bit for bit, gimage to the atomic order);
    a loss on the residual only, on warped and residual together, and the gt gradient."""
    img, flow, gt, gw, gr = _warp_case(_seed("fp32", align, shape), *shape)
    what = f"align={align} {shape}"
    cases = [(("image", "flow"), None, gw, None), (("image",), None, gw, None), (("flow",), None, gw, None),
             (("image", "flow", "gt"), gt, None, gr), (("image", "flow", "gt"), gt, gw, gr), (("gt",), gt, gw, gr),
             (("flow",), gt, None, gr)]
    both = None
    for want, g_t, g_w, g_r in cases:
        ref = _backwarp_ref(orc, img, flow, g_t, align, g_w, g_r, want)
        truth = _backwarp_ref(orc, img.double(), flow.double(), None if g_t is None else g_t.double(), align,
                              None if g_w is None else g_w.double(), None if g_r is None else g_r.double(), want)
        got = _backwarp_cuda(dcb, img, flow, g_t, align, g_w, g_r, want)
        _check_warp(got, ref, want, 1e-5, f"{what} {want} gt={g_t is not None} gw={g_w is not None} gr={g_r is not None}", truth)
        if g_t is None and len(want) == 2:
            both = got
        elif g_t is None:
            k = want[0]
            if k == "flow":
                assert torch.equal(got[2]["flow"], both[2]["flow"]), f"{what}: gflow alone vs both gradients"
            else:
                assert_close(got[2]["image"], both[2]["image"], 1e-6, f"{what}: gimage alone vs both gradients")


@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=str)
def test_backwarp_huge_and_nonfinite_flows(dcb, orc, align, dtype):
    """Huge finite flows (+-4000, 1e9) are ordinary flows whose taps leave the frame: the reference's values. A non-finite
    flow (NaN, +-inf) is the library's documented departure: the pixel warps to 0 and scatters nothing (torch's grid_sample
    gives platform-dependent results for a NaN grid, so no value is pinned there). Checked as: warped == 0 there, gimage
    equal to the reference with those flows moved far out of the frame (finite everywhere), and gflow finite and equal to
    the reference at every pixel whose flow is finite."""
    n, c, h, w = 2, 3, 18, 33
    img, flow, _, gw, _ = _warp_case(_seed("huge", align, dtype), n, c, h, w)
    img, flow, gw = img.to(dtype), flow.to(dtype), gw.to(dtype)
    rel = 1e-5 if dtype == torch.float32 else 1e-12
    big = flow.clone()
    big[0, 0, 2:4, 5:9] = 4000.0; big[0, 1, 6, :] = -4000.0; big[1, 0, 9, 10:20] = 1e9; big[1, 1, 11, 3] = -1e9
    big[1, 0, 12:14, :] = -4000.0
    big[0, 0, 14, 1] = -(1 + 0.25)                              # a tap half outside the left edge
    want = ("image", "flow")
    ref = _backwarp_ref(orc, img, big, None, align, gw, None, want)
    truth = None if dtype == torch.float64 else _backwarp_ref(orc, img.double(), big.double(), None, align, gw.double(), None, want)
    got = _backwarp_cuda(dcb, img, big, None, align, gw, None, want)
    _check_warp(got, ref, want, rel, f"huge flows {dtype} align={align}", truth)

    bad = flow.clone()
    bad[0, 0, 3, 4] = float("nan"); bad[0, 1, 7, 20:25] = float("nan"); bad[1, 0, 5, :] = float("inf")
    bad[1, 1, 10:12, 30] = -float("inf"); bad[1, :, 15, 15] = float("nan")
    nonfinite = ~torch.isfinite(bad).all(1)                  # [n, h, w]
    got = _backwarp_cuda(dcb, img, bad, None, align, gw, None, want)
    warped, gimage, gflow = got[0].cpu(), got[2]["image"].cpu(), got[2]["flow"].cpu()
    assert (warped.permute(1, 0, 2, 3)[:, nonfinite] == 0).all(), "a non-finite flow warps to 0"
    assert torch.isfinite(gimage).all(), "a non-finite flow scatters nothing into gimage"
    fin = ~nonfinite
    assert torch.isfinite(gflow.permute(1, 0, 2, 3)[:, fin]).all(), "gflow is finite wherever the flow is"
    far = torch.where(torch.isfinite(bad), bad, torch.full_like(bad, 1e9))     # taps far out of the frame: the same contract
    ref = _backwarp_ref(orc, img, far, None, align, gw, None, want)
    truth = None if dtype == torch.float64 else _backwarp_ref(orc, img.double(), far.double(), None, align, gw.double(), None, want)
    sel = lambda t: t.permute(1, 0, 2, 3)[:, fin]
    assert_close(sel(warped), sel(ref[0]), rel, "non-finite: warped elsewhere", truth=None if truth is None else sel(truth[0]))
    assert_close(gimage, ref[2]["image"], rel, "non-finite: gimage", truth=None if truth is None else truth[2]["image"])
    assert_close(sel(gflow), sel(ref[2]["flow"]), rel, "non-finite: gflow elsewhere",
                 truth=None if truth is None else sel(truth[2]["flow"]))


# ---------------------------------------------------------------------------------------------------------------------
# D. 64-bit offset forms, GPU against GPU
# ---------------------------------------------------------------------------------------------------------------------
def _free_device_memory():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def test_splat_backward_wide_gradient_view(dcb, impl):
    """A grad_out view with strides (., 64, 2**30, 1) spans 2**30 + 63 elements per plane: the generic source pass takes
    64-bit offsets (k_bwd_source<T, TF, long long>). Only the index type differs from the run on the .contiguous() copy,
    so the gradients are the same bits. fp16 has no 64-bit form and refuses such a view (DCB_E_LIMIT -> ValueError)
    rather than fall back. One 4 GiB buffer serves every dtype; it is released at the end."""
    n, c, h, w = 1, 4, 2, 64
    L = dcb._lib
    sizes, strides = (n, c, h, w), (c * 64, 64, 1 << 30, 1)
    need = (c - 1) * 64 + (h - 1) * (1 << 30) + w               # elements the view reaches
    buf = torch.empty(need * 4, dtype=torch.uint8, device="cuda")
    wide = None
    try:
        tin, flow, metric, gout = make_inputs(17, n, c, h, w, flow_scale=0.6)
        for dtype, flow_dtype in ((torch.bfloat16, torch.float32), (torch.bfloat16, torch.bfloat16), (torch.float32, torch.float32)):
            for mode, lmode in (("sum", L.MODE_SUM), ("soft", L.MODE_SOFT)):
                ti, fl, g = tin.cuda().to(dtype), flow.cuda().to(flow_dtype), gout.cuda().to(dtype)
                me = metric.cuda().to(dtype) if mode == "soft" else None
                wide = torch.as_strided(buf.view(dtype), sizes, strides)
                wide.copy_(g)
                out, norm = impl._forward(ti, fl, me, None, lmode, L.EPS_ADD, False, True)
                need_grads = (True, True, me is not None)
                a = impl._backward(wide, ti, fl, me, out, norm, None, lmode, L.EPS_ADD, need_grads)
                b = impl._backward(wide.contiguous(), ti, fl, me, out, norm, None, lmode, L.EPS_ADD, need_grads)
                for k, x, y in zip(NAMES, a, b):
                    if y is None:
                        assert x is None
                        continue
                    assert torch.equal(x, y), f"{dtype} flow {flow_dtype} {mode}: grad {k} with 64-bit offsets differs"
                assert a[0].abs().sum() > 0 and a[1].abs().sum() > 0
        # fp16: refused, not computed some other way
        ti, fl = tin.cuda().half(), flow.cuda()
        wide = torch.as_strided(buf.view(torch.float16), sizes, strides)
        wide.copy_(gout.cuda().half())
        for lmode, me in ((L.MODE_SUM, None), (L.MODE_SOFT, metric.cuda().half())):
            out, norm = impl._forward(ti, fl, me, None, lmode, L.EPS_ADD, False, True)
            with pytest.raises(ValueError, match="2\\^30"):
                impl._backward(wide, ti, fl, me, out, norm, None, lmode, L.EPS_ADD, (True, True, me is not None))
        torch.cuda.synchronize()
    finally:
        del buf, wide                                          # the view keeps the storage alive too
        _free_device_memory()


def test_backwarp_image_view_with_64bit_offsets(dcb):
    """A bf16 image view with strides (., 64, 2**30, 1) over 3 rows reaches element 2**31 + 127: its offsets need 64 bits
    (the paired-rows kernel refuses it, the generic kernels take it). Forward, residual and gflow equal the run on the
    .contiguous() copy bit for bit; gimage (atomics) to 1e-6. The 4 GiB buffer is released at the end."""
    n, c, h, w = 1, 2, 3, 64
    sizes, strides = (n, c, h, w), (c * 64, 64, 1 << 30, 1)
    need = (c - 1) * 64 + (h - 1) * (1 << 30) + w
    assert need - 1 >= 1 << 31
    buf = torch.empty(need, dtype=torch.bfloat16, device="cuda")
    view = None
    try:
        g = torch.Generator().manual_seed(29)
        img = torch.rand(n, c, h, w, generator=g).cuda().bfloat16()
        flow = (torch.randn(n, 2, h, w, generator=g) * 1.2).cuda()
        gt = torch.rand(n, c, h, w, generator=g).cuda().bfloat16()
        gw = torch.randn(n, c, h, w, generator=g).cuda().bfloat16()
        gr = torch.randn(n, c, h, w, generator=g).cuda().bfloat16()
        view = torch.as_strided(buf, sizes, strides)
        view.copy_(img)
        for align in (False, True):
            res = []
            for im in (view, img):
                ii, ff = im.detach().requires_grad_(True), flow.clone().requires_grad_(True)
                warped, residual = dcb.backwarp_residual(ii, ff, gt, align_corners=align)
                gi, gf = torch.autograd.grad([warped, residual], [ii, ff], [gw, gr])
                res.append((warped, residual, gi, gf))
            (w1, r1, gi1, gf1), (w2, r2, gi2, gf2) = res
            assert torch.equal(w1, w2) and torch.equal(r1, r2), f"align={align}: forward with 64-bit offsets differs"
            assert torch.equal(gf1, gf2), f"align={align}: gflow with 64-bit offsets differs"
            assert_close(gi1.float(), gi2.float(), 1e-6, f"align={align}: gimage with 64-bit offsets")
            assert w1.abs().sum() > 0 and gi1.abs().sum() > 0
        torch.cuda.synchronize()
    finally:
        del buf, view
        _free_device_memory()


# ---------------------------------------------------------------------------------------------------------------------
# E. Fusion backward
# ---------------------------------------------------------------------------------------------------------------------
def _fuse_inputs(seed, n=2, c=12, h=20, w=28):
    """Confidences of both signs, exactly 0 on one side (rows 0..3: conf_a, rows 4..7: conf_b) and on both sides (rows 8..9),
    and a double-hole block (rows 12..15, cols 4..11)."""
    g = torch.Generator().manual_seed(seed)
    A, B = torch.randn(n, c, h, w, generator=g), torch.randn(n, c, h, w, generator=g)
    ca, cb = torch.randn(n, 1, h, w, generator=g), torch.randn(n, 1, h, w, generator=g)
    ca[:, :, 0:4] = 0.0
    cb[:, :, 4:8] = 0.0
    ca[:, :, 8:10] = 0.0; cb[:, :, 8:10] = 0.0
    oa = (torch.rand(n, 1, h, w, generator=g) > 0.6).float(); ob = (torch.rand(n, 1, h, w, generator=g) > 0.6).float()
    oa[:, :, 12:16, 4:12] = 1.0; ob[:, :, 12:16, 4:12] = 1.0
    return A, B, ca, cb, oa, ob


FUSE_NAMES = ("A", "B", "conf_a", "conf_b")


def _assert_fuse_grad(k, got, ref, ca, cb, what):
    """A confidence gradient is about gw / 1e-6 where both clamped confidences are 0 (the normaliser is the 1e-6 alone) and
    O(1) elsewhere. Each set is compared on its own scale, so that a tolerance scaled by the amplified pixels cannot hide an
    error at the ordinary ones."""
    if not k.startswith("conf"):
        assert_close(got, ref, 1e-5, f"{what} grad {k}")
        return
    tiny = ((ca.clamp(min=0) + cb.clamp(min=0)) < 1e-3).expand_as(ref)
    assert tiny.any() and (~tiny).any()
    got = got.cpu()
    assert_close(got[tiny], ref[tiny], 1e-5, f"{what} grad {k}, normaliser 1e-6")
    assert_close(got[~tiny], ref[~tiny], 1e-5, f"{what} grad {k}, ordinary pixels")


@pytest.mark.parametrize("occ", [True, False])
@pytest.mark.parametrize("c", [3, 12])
def test_fuse_gradient_subsets(dcb, orc, occ, c):
    """Every non-empty subset of {A, B, conf_a, conf_b} (the need_w skip when no confidence gradient is wanted), with and
    without occlusion masks: the oracle's gradients, None for the others. clamp(min=0) passes the gradient at a confidence
    of exactly 0 (one side or both), and the double holes give confidence gradients of exactly 0."""
    A, B, ca, cb, oa, ob = _fuse_inputs(_seed("fuse", occ, c), c=c)
    go = torch.randn(A.shape, generator=torch.Generator().manual_seed(5))
    for r in range(1, 5):
        for want in itertools.combinations(FUSE_NAMES, r):
            cpu = [t.clone().requires_grad_(k in want) for k, t in zip(FUSE_NAMES, (A, B, ca, cb))]
            ref = orc.fuse(*cpu, oa if occ else None, ob if occ else None)
            ref.backward(go)
            gpu = [t.cuda().requires_grad_(k in want) for k, t in zip(FUSE_NAMES, (A, B, ca, cb))]
            got = dcb.bidir_fuse(*gpu, oa.cuda() if occ else None, ob.cuda() if occ else None)
            got.backward(go.cuda())
            what = f"fuse occ={occ} C={c} {want}"
            assert_close(got, ref, 1e-5, f"{what} fused")
            for k, a, b in zip(FUSE_NAMES, gpu, cpu):
                if k not in want:
                    assert a.grad is None, f"{what}: grad {k} was not asked for"
                    continue
                _assert_fuse_grad(k, a.grad, b.grad, ca, cb, what)
                if k.startswith("conf"):
                    gc = a.grad.cpu()
                    zero_rows = slice(0, 4) if k == "conf_a" else slice(4, 8)
                    assert (gc[:, :, zero_rows] != 0).any() and (gc[:, :, 8:10] != 0).any(), \
                        f"{what}: clamp(min=0) passes the gradient at a confidence of exactly 0"
                    if occ:
                        assert (gc[:, :, 12:16, 4:12] == 0).all(), f"{what}: double holes give a zero confidence gradient"
