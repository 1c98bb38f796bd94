"""The forward splat on exactly representable inputs: bit for bit against the fp64 oracle, no tolerance.

The forward scatter merges corner pieces in registers before they reach the accumulators (csrc/splat_pipe.cu scatter_strip:
east pieces handed to the right lane, the south piece carried down the strip, and on rough flow the diagonal hand-overs and
three vertical joins; the recipe rider repeats every merge on two more channels; csrc/splat_planar.cuh has a third copy).
A dropped, doubled or misplaced piece of weight 1/64 can hide under a tolerance scaled by the tensor's maximum, so these
tests take inputs on which fp32 arithmetic is exact:

  * data are small integers (|v| <= 8), flow components multiples of 1/8 (|flow| < 32, so bf16 / fp16 flows are exact too),
    the `linear` metric is in {1/2, 1, 2, 3}, a mask factor a multiple of 1/8;
  * then x + flow is exact, the corner weights are multiples of 1/64, every piece v * g * w is exact (a multiple of 1/128),
    and as long as every partial sum stays below 2^17 in magnitude every fp32 addition is exact in ANY order: register
    merges, L2 reductions, list gathers and shared-memory sums all give the one exact value (the bound is checked on the
    host, test_exactness_bound).

So in `sum` mode every forward family returns exactly the fp64 oracle cast to the output dtype; in `avg` / `linear` the
normaliser (with the zeroeps rule) is exact and the output is one reciprocal and one multiply, within 2 fp32 ulps of the
fp64 value (1 ulp of a bf16 / fp16 output). The sum-mode backward is exact as well (dyadic upstream gradient).

The flow fields are built so that every merge event fires, at the geometry edges where it can go wrong; a numpy model of
the pipe kernel's strip geometry counts the events, and a CPU test keeps those counts above a floor, so the suite notices if
the generator or the kernel's geometry drifts. The recipe rider is checked as a number through its occlusion masks with a
constant rider (section 3 below)."""
import contextlib
import importlib
import itertools

import numpy as np
import pytest
import torch

# ---------------------------------------------------------------------------------------------------------------------
# strip geometry of the pipe kernel, copied from csrc/splat_pipe.cu (k_splat_step / scatter_strip / splat_pipe_impl)
# ---------------------------------------------------------------------------------------------------------------------
LANES = 32             # one warp per strip column: lane i is column 32 * tx + i
K_ROWS = 4             # kRows: rows loaded at once; rough_pass is decided per group of kRows rows
K_PASSES = 2           # kPasses: row groups per full-height strip (the vertical carry spans them)
K_STRIP_H = K_ROWS * K_PASSES
K_ROUGH_LANES = 5      # kRoughLanes: lanes whose flow jumps by more than ROUGH_JUMP make a rough group
ROUGH_JUMP = 0.25
DEAD = -7              # kDead: key of a dead footprint

EVENT_FLOOR = 50
EVENTS = ("abut_plain", "abut_rough", "t_dn", "t_up", "join_plain", "join_rough", "join_e", "join_s", "switch_carry",
          "lane31_take", "strip_seam", "dead_lane", "dead_in_chain", "single_pass", "ragged_group",
          "x0_left", "x0_right", "y0_top", "y0_bottom")


def strip_rows(h, tail_percent=0):
    """(first row, passes) of every strip row of a frame, as splat_pipe_impl sets ny_big / tiles_y and k_splat_step maps
    blockIdx.y (the rider passes use tail_percent = 0)."""
    rows_fine = (h * tail_percent // 100) // K_STRIP_H * K_STRIP_H
    ny_big = (h - rows_fine) // K_STRIP_H
    rest = h - ny_big * K_STRIP_H
    tiles_y = ny_big + (rest + K_ROWS - 1) // K_ROWS
    return [(by * K_STRIP_H, K_PASSES) if by < ny_big else (ny_big * K_STRIP_H + (by - ny_big) * K_ROWS, 1)
            for by in range(tiles_y)]


def pipe_events(flow, tail_percent=0):
    """Count the register-merge events of scatter_strip on `flow` ([N,2,H,W] numpy): which lanes hand over / join, in which
    form, at which geometry edge. Only counts; the numerical reference is the fp64 oracle."""
    flow = np.asarray(flow, dtype=np.float32)
    n, _, h, w = flow.shape
    tiles_x = (w + LANES - 1) // LANES
    pitch = w + 2
    lane = np.arange(LANES)[None, :]
    x = np.arange(tiles_x)[:, None] * LANES + lane                       # [tiles_x, 32]
    xin = x < w
    xs = np.where(xin, x, 0)
    cnt = dict.fromkeys(EVENTS, 0)
    with np.errstate(invalid="ignore", over="ignore"):
        for f in range(n):
            for y_first, passes in strip_rows(h, tail_percent):
                pend_key = np.full(x.shape, DEAD)
                pend_ok = np.zeros(x.shape, bool)
                prev_rough = None
                for p in range(passes):
                    yb = y_first + p * K_ROWS
                    if yb >= h:
                        break
                    rows = min(K_ROWS, h - yb)
                    fx0 = np.where(xin, flow[f, 0, yb, xs], 0).astype(np.float32)
                    fy0 = np.where(xin, flow[f, 1, yb, xs], 0).astype(np.float32)
                    jump = (lane > 0) & ((np.abs(fx0 - np.roll(fx0, 1, 1)) > ROUGH_JUMP) | (np.abs(fy0 - np.roll(fy0, 1, 1)) > ROUGH_JUMP))
                    rough = (jump.sum(1) >= K_ROUGH_LANES)[:, None]             # per strip column
                    for r in range(K_ROWS):
                        y = yb + r
                        in_img = xin & (r < rows)
                        fl_x = np.where(in_img, flow[f, 0, min(y, h - 1), xs], 0).astype(np.float32)
                        fl_y = np.where(in_img, flow[f, 1, min(y, h - 1), xs], 0).astype(np.float32)
                        fx = x.astype(np.float32) + fl_x
                        fy = np.float32(y) + fl_y
                        finite = np.isfinite(fx) & np.isfinite(fy) & (np.abs(fx) < 3.0e38) & (np.abs(fy) < 3.0e38)
                        x0 = np.where(finite, np.floor(np.where(finite, fx, 0)), -(1 << 40)).astype(np.int64)
                        y0 = np.where(finite, np.floor(np.where(finite, fy, 0)), -(1 << 40)).astype(np.int64)
                        alive = in_img & finite & (x0 >= -1) & (x0 <= w - 1) & (y0 >= -1) & (y0 <= h - 1)
                        key = np.where(alive, (y0 + 1) * pitch + (x0 + 1), DEAD)
                        lkey = np.roll(key, 1, 1)
                        nb = (lane > 0) & alive & (lkey != DEAD)
                        t_ab = nb & (lkey + 1 == key)
                        t_dn = nb & (lkey + 1 + pitch == key) & rough
                        t_up = nb & (lkey + 1 - pitch == key) & rough
                        join = (pend_key == key) & alive
                        join_e = (pend_key == key + 1) & alive & rough
                        join_s = (pend_key == key + pitch) & alive & rough
                        cnt["abut_plain"] += int((t_ab & ~rough).sum())
                        cnt["abut_rough"] += int((t_ab & rough).sum())
                        cnt["t_dn"] += int(t_dn.sum())
                        cnt["t_up"] += int(t_up.sum())
                        cnt["join_plain"] += int((join & ~rough).sum())
                        cnt["join_rough"] += int((join & rough).sum())
                        cnt["join_e"] += int(join_e.sum())
                        cnt["join_s"] += int(join_s.sum())
                        any_join = join | join_e | join_s
                        if r == 0 and p > 0:
                            cnt["switch_carry"] += int((any_join & (rough != prev_rough)).sum())
                        took = t_ab | t_dn | t_up
                        cnt["lane31_take"] += int(took[:, LANES - 1].sum())
                        # lane 31 and lane 0 of the next strip column: footprints that abut, which must NOT be handed over
                        seam = alive[:-1, LANES - 1] & alive[1:, 0] & (key[1:, 0] == key[:-1, LANES - 1] + 1)
                        cnt["strip_seam"] += int(seam.sum())
                        cnt["dead_lane"] += int((alive & (x == w - 1) & (x % LANES != LANES - 1)).sum())
                        cnt["dead_in_chain"] += int((pend_ok & in_img & ~alive).sum())
                        if passes == 1:
                            cnt["single_pass"] += int((took | any_join).sum())
                        if rows < K_ROWS:
                            cnt["ragged_group"] += int((took | any_join).sum())
                        cnt["x0_left"] += int((alive & (x0 == -1)).sum())
                        cnt["x0_right"] += int((alive & (x0 == w - 1)).sum())
                        cnt["y0_top"] += int((alive & (y0 == -1)).sum())
                        cnt["y0_bottom"] += int((alive & (y0 == h - 1)).sum())
                        pend_key = np.where(alive, key + pitch, DEAD)
                        pend_ok = alive & (x0 >= 0) & (y0 < h - 1)
                    prev_rough = rough
    return cnt


# ---------------------------------------------------------------------------------------------------------------------
# dyadic flow fields
# ---------------------------------------------------------------------------------------------------------------------
# per 4-row group: rough (R) or smooth (S) first row; every 16-row strip holds an R -> S and an S -> R switch
GROUP_STYLE = "RSRRSSRSRSSR"


def dyadic_flow(seed, n, h, w, far=True, dead=True):
    """[N,2,H,W] float64 flow whose components are multiples of 1/8 with |flow| < 32 (non-finite / huge at dead pixels).

    Every pixel gets an integer offset in {-1, 0, 1}^2 on top of a fractional part in {0, 1/8, ..., 7/8} (0 included: some
    landings are integer, some corner weights zero), so neighbouring lanes and consecutive rows fall into every relation of
    the merges: abutting, one right and one down / up, the same footprint, one row down and one cell left, no relation.
    The first row of a group decides rough_pass: in smooth groups (GROUP_STYLE) it carries one offset with fractional
    jitter of at most 1/8, and the group's other rows are half smooth, half rough. Columns and rows at the frame edges
    are pushed half outside, a few sources come from about 30 px away, and a few pixels are NaN, +inf or 1e9."""
    rng = np.random.default_rng(seed)
    frac = rng.integers(0, 8, size=(n, 2, h, w)) / 8.0
    off = rng.integers(-1, 2, size=(n, 2, h, w)).astype(np.float64)
    flow = off + frac
    for g0 in range(0, h, K_ROWS):
        if GROUP_STYLE[(g0 // K_ROWS) % len(GROUP_STYLE)] == "S":
            base = rng.integers(-1, 2, size=(n, 2, 1, 1)) + rng.integers(0, 7, size=(n, 2, 1, 1)) / 8.0
            jitter = rng.integers(0, 2, size=(n, 2, K_ROWS, w)) / 8.0
            smooth = base + jitter
            rows = min(K_ROWS, h - g0)
            flow[:, :, g0] = smooth[:, :, 0]
            keep = rng.random((n, 1, rows - 1, w)) < 0.5
            flow[:, :, g0 + 1:g0 + rows] = np.where(keep, smooth[:, :, 1:rows], flow[:, :, g0 + 1:g0 + rows])
    # frame edges: footprints with x0 = -1 / W-1 and y0 = -1 / H-1
    # (the two outermost columns / rows land at -1 + k/8 or at size - 1 + k/8 with 60 % probability)
    yy, xx = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    for c, pos, size in ((0, xx, w), (1, yy, h)):
        k = rng.integers(1, 8, size=(n, h, w)) / 8.0
        pick = rng.random((n, h, w)) < 0.6
        flow[:, c] = np.where(pick & (pos < 2), -1 - pos + k, flow[:, c])
        flow[:, c] = np.where(pick & (pos >= size - 2), size - 1 - pos + k, flow[:, c])
    if far:
        m = rng.random((n, 1, h, w)) < 0.02
        flow = np.where(m, rng.choice([-30.0, 29.0], size=(n, 2, h, w)) + frac, flow)
    if dead:
        m = rng.random((n, 1, h, w)) < 0.012
        flow[:, :1] = np.where(m, rng.choice([np.nan, np.inf, 1e9], size=(n, 1, h, w)), flow[:, :1])
    return flow


def dyadic_data(seed, shape, lo=-8, hi=8):
    return np.random.default_rng(seed).integers(lo, hi + 1, size=shape).astype(np.float64)


def dyadic_metric(seed, n, h, w):
    return np.random.default_rng(seed).choice([0.5, 1.0, 2.0, 3.0], size=(n, 1, h, w))


# the pipeline field: W not a multiple of 32 (dead lanes), H not a multiple of 16 or 4 (single-pass strips, a ragged group)
PIPE_SHAPE = (3, 45, 200)
TAIL_PERCENT = 60


def _exact_bound(orc, data, flow, g=None):
    """Largest partial sum the scatter can form: the fp64 oracle's splat of |v| * |g| (and of |g|, the weight channel)."""
    a = np.abs(data) * (1.0 if g is None else np.abs(g))
    planes = [a] if g is None else [a, np.abs(g)]
    return max(float(np.nanmax(orc.splat_fwd(np.ascontiguousarray(p), np.ascontiguousarray(flow)))) for p in planes)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the fields reach every merge event, and stay in the exact range
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tail_percent", [0, TAIL_PERCENT])
def test_pipe_field_reaches_every_merge_event(tail_percent):
    n, h, w = PIPE_SHAPE
    cnt = pipe_events(dyadic_flow(1, n, h, w), tail_percent)
    low = {k: v for k, v in cnt.items() if v < EVENT_FLOOR}
    assert not low, f"merge events below {EVENT_FLOOR} on the exact-test field: {low} (all counts: {cnt})"


def test_rider_field_reaches_every_merge_event():
    n, h, w = RIDER_SHAPE
    cnt = pipe_events(rider_flows(2, n, h, w, RIDER_U[torch.float32])[0])
    low = {k: v for k, v in cnt.items() if v < EVENT_FLOOR}
    assert not low, f"rider field: merge events below {EVENT_FLOOR}: {low} (all counts: {cnt})"


def test_exactness_bound():
    """Every partial sum of the exact tests stays below 2^17: fp32 additions of multiples of 1/128 are then exact."""
    from oracle import oracle as orc
    n, h, w = PIPE_SHAPE
    flow = dyadic_flow(1, n, h, w)
    for c in (1, 3, 16):
        data = dyadic_data(2, (n, c, h, w))
        assert _exact_bound(orc, data, flow, dyadic_metric(3, n, h, w)) < 2.0 ** 17
    # the dyadic grid: every finite flow component a multiple of 1/8 below 32 in magnitude, every metric a multiple of 1/2
    fin = flow[np.isfinite(flow) & (np.abs(flow) < 1e6)]
    assert np.all(fin * 8 == np.round(fin * 8)) and np.abs(fin).max() < 32
    dead = ~np.isfinite(flow[:, 0]) | (np.abs(flow[:, 0]) > 1e6)
    assert 0.005 < dead.mean() < 0.03


# ---------------------------------------------------------------------------------------------------------------------
# section 3: the rider of the conditioning recipe, checked through bit-equal masks
# ---------------------------------------------------------------------------------------------------------------------
# flow2 == U = (-u, u) in even frames and (u, -u) in odd ones (a rider constant per frame, each component a power of two in magnitude; the signs differ so that a piece
# that lands in the wrong rider channel shows too), flow1 = -U + delta with delta in
# {-1/4, 0, 1/4}^2. Every rider piece is then U times the weight channel's piece, so the normalised rider is U at every
# covered target whatever the merges did -- provided the rider merges do what the weight-channel merges do -- and the mask
# of compute_mask(flow2, flow1) at target t is exactly [||delta_t|| > 0.3] (||delta|| is 0, 0.25 or 0.354: at least 0.05
# from the threshold). A piece of weight w dropped or doubled in rider channel c at t moves component c of the compared
# vector by (w / S_t) * U_c (S_t: the normaliser), and w >= 1/16. bf16 keeps |flow| <= 32.25 on its 8-bit significand, so
# u = 32 there. Sources move right and up by u in even frames (the bottom rows, with their single-pass strips and ragged
# group, stay in the frame), left and down in odd frames (the last strip column, with its dead lanes, stays in the frame); the
# frame is tall and wide enough that much of it stays covered.
RIDER_SHAPE = (2, 141, 230)
RIDER_U = {torch.float32: 64.0, torch.bfloat16: 32.0}
RIDER_MARGIN = 0.05


def rider_flows(seed, n, h, w, u, far_dead=True):
    """(flow1, flow2) of the rider tests as float64 numpy: flow2 = (-u, u) in even frames and (u, -u) in odd
    ones, flow1 = -flow2 + delta."""
    rng = np.random.default_rng(seed)
    delta = rng.integers(-1, 2, size=(n, 2, h, w)) / 4.0
    for g0 in range(0, h, K_ROWS):                 # smooth groups: the first row jumps by at most 1/4
        if GROUP_STYLE[(g0 // K_ROWS) % len(GROUP_STYLE)] == "S":
            delta[:, :, g0] = rng.integers(0, 2, size=(n, 2, w)) / 4.0
    flow2 = np.full((n, 2, h, w), u)
    flow2[0::2, 0] = -u
    flow2[1::2, 1] = -u
    flow1 = delta - flow2
    if far_dead:
        m = rng.random((n, 1, h, w)) < 0.01
        flow1[:, :1] = np.where(m, 1e9, flow1[:, :1])
    return flow1, flow2


def rider_sensitivity(flow1, flow2):
    """Per target: covered (normaliser > 0), ||delta_t||, and per rider channel c whether a piece dropped, doubled or
    misplaced in that channel alone must flip the mask: the smallest nonzero piece over the normaliser, times |U_c|,
    exceeds 0.3 + ||delta_t|| by RIDER_MARGIN. Returns (covered, sensitive [2, N, H, W], delta)."""
    from oracle import oracle as orc
    n, _, h, w = flow1.shape
    norm = orc.splat_fwd(np.ones((n, 1, h, w)), flow1)[:, 0]
    # the smallest nonzero corner weight reaching a target, bounded by the grid: delta in {-1/4, 0, 1/4} makes every
    # nonzero corner weight >= 1/16
    wmin = 1.0 / 16
    u = flow2[:, :, 0, 0]                                            # the constant rider, per frame and channel
    delta = np.linalg.norm(flow1 + flow2, axis=1)
    covered = norm > 0
    shift = wmin / np.where(covered, norm, 1.0)
    sensitive = np.stack([covered & (delta < 0.3) & (shift * np.abs(u[:, c, None, None]) > 0.3 + delta + RIDER_MARGIN)
                          for c in range(2)])
    return covered, sensitive, delta


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_rider_bound(dtype):
    """The constant-rider field is where the mask test can see a rider merge bug: all masks 0.05 away from the threshold,
    and at (nearly) every covered target with mask 0 a single wrong piece in EITHER rider channel must flip the mask."""
    n, h, w = RIDER_SHAPE
    u = RIDER_U[dtype]
    flow1, flow2 = rider_flows(2, n, h, w, u)
    assert np.all(np.abs(flow2) == u) and np.all(flow2[:, 0] == -flow2[:, 1]) and np.log2(u) == int(np.log2(u))
    covered, sensitive, delta = rider_sensitivity(flow1, flow2)
    fin = np.isfinite(delta) & (delta < 1)
    assert np.all(np.abs(delta[fin] - 0.3) >= RIDER_MARGIN - 1e-12)
    zero = covered & (delta < 0.3)
    assert zero.sum() > 0.4 * covered.sum() and covered.mean() > 0.25
    for c in range(2):
        assert sensitive[c].sum() >= 0.97 * zero.sum(), \
            f"rider channel {c}: {int(sensitive[c].sum())} of {int(zero.sum())} mask-0 targets sensitive"
    if dtype == torch.bfloat16:      # every flow value exact in bf16
        f = torch.from_numpy(flow1[np.abs(flow1) < 1e6])
        assert torch.equal(f.to(torch.bfloat16).double(), f)


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dcb():
    import diffcodec_b200
    return diffcodec_b200


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    oracle.lib()
    return oracle


OPTION_DEFAULTS = {"fwd_path": 0, "pipe_group_bytes": 0, "pipe_ring_slots": 1, "pipe_tail_percent": -1, "lists_nhwc": 1,
                   "planar_one_launch": 0}


@contextlib.contextmanager
def options(dcb, **opts):
    """Library options for the block; every option touched is back at its default afterwards and the workspaces sized
    under it are released."""
    L = dcb._lib
    try:
        for k, v in opts.items():
            L.set_option(k, v)
        L.release_workspaces()
        yield
    finally:
        for k in opts:
            L.set_option(k, OPTION_DEFAULTS[k])
        L.release_workspaces()


def _orc_fwd(orc, data, flow, mode, metric=None, mask=None):
    """(out, normaliser) in fp64 numpy: the oracle's sum-splat of [in * g, g] (g: 1 for avg, the metric for linear); the
    zeroeps rule; the (1 - mask) factor."""
    if mode == "sum":
        out, norm = orc.splat_fwd(data, flow), None
    else:
        g = np.ones_like(data[:, :1]) if mode == "avg" else metric
        acc = orc.splat_fwd(np.concatenate([data * g, g], 1), flow)
        norm = np.where(acc[:, -1:] == 0, 1.0, acc[:, -1:])
        out = acc[:, :-1] / norm
    if mask is not None:
        out = out * (1 - mask)
    return out, norm


def _ulp(x, dtype):
    bits = {torch.float32: 23, torch.bfloat16: 7, torch.float16: 10, torch.float64: 52}[dtype]
    a = np.abs(x)
    return np.where(a > 0, np.exp2(np.floor(np.log2(np.where(a > 0, a, 1.0))) - bits), 0.0)


def _where(bad, shape):
    i = int(np.flatnonzero(bad)[0])
    return tuple(int(v) for v in np.unravel_index(i, shape))


# strip layouts for failure messages: (name, pipe_tail_percent, rough form). The planar pipeline scatters single-pass
# 32 x 4 strips in the plain form only (csrc/splat_planar.cuh): the layout of a 100 % tail without the rough form.
PIPE_GEOM = ("accumulator pipeline", 0, True)
PIPE_TAIL_GEOM = ("accumulator pipeline with a single-pass tail", TAIL_PERCENT, True)
PLANAR_GEOM = ("planar pipeline", 100, False)


def merges_at(flow, f, y, x, geom=PIPE_GEOM):
    """The sources whose footprint covers target (y, x) of frame f, each with the register merges the strip layout `geom`
    applies to it (relation to the lane on its left and to the row above it in its strip, and the form of its row group):
    what a failure message names next to the wrong pixel. Families with other kernels are described in the pipeline's
    layout, which the message says."""
    fl = np.asarray(flow[f], dtype=np.float64)
    h, w = fl.shape[1:]
    pitch = w + 2
    name, tail_percent, rough_form = geom
    first_row = np.zeros(h, np.int64)              # first row of the strip holding each row
    for y_first, passes in strip_rows(h, tail_percent):
        first_row[y_first:y_first + passes * K_ROWS] = y_first

    def foot(sy, sx):
        fx, fy = sx + fl[0, sy, sx], sy + fl[1, sy, sx]
        if not (np.isfinite(fx) and np.isfinite(fy) and abs(fx) < 3e38 and abs(fy) < 3e38):
            return None
        x0, y0 = int(np.floor(fx)), int(np.floor(fy))
        return (x0, y0) if -1 <= x0 <= w - 1 and -1 <= y0 <= h - 1 else None

    def key(p):
        return None if p is None else (p[1] + 1) * pitch + p[0] + 1

    out = []
    with np.errstate(invalid="ignore", over="ignore"):
        for sy in range(h):
            for sx in range(w):
                p = foot(sy, sx)
                if p is None or p[0] not in (x - 1, x) or p[1] not in (y - 1, y):
                    continue
                k, lane = key(p), sx % LANES
                yb = first_row[sy] + (sy - first_row[sy]) // K_ROWS * K_ROWS     # first row of the row group
                x_lo = sx - lane
                row0 = np.zeros((2, LANES))              # lanes beyond the frame load a zero flow
                row0[:, :min(LANES, w - x_lo)] = fl[:, yb, x_lo:x_lo + LANES]
                rough = rough_form and int(((np.abs(np.diff(row0, axis=1)) > ROUGH_JUMP).any(0)).sum()) >= K_ROUGH_LANES
                rel = []
                kl = key(foot(sy, sx - 1)) if lane > 0 else None
                if kl is not None:
                    rel += [n for n, d in (("abut", 1), ("t_dn", 1 + pitch), ("t_up", 1 - pitch)) if kl + d == k
                            and (n == "abut" or rough)]
                ka = key(foot(sy - 1, sx)) if sy > first_row[sy] else None        # the carry stays inside a strip
                if ka is not None:
                    rel += [n for n, d in (("join", 0), ("join_e", 1), ("join_s", pitch)) if ka + pitch == k + d
                            and (n == "join" or rough)]
                kr = key(foot(sy, sx + 1)) if lane < LANES - 1 and sx + 1 < w else None
                if kr is not None:
                    rel += [n for n, d in (("gives abut", 1), ("gives t_dn", 1 + pitch), ("gives t_up", 1 - pitch))
                            if k + d == kr and (n == "gives abut" or rough)]
                out.append(f"source (y={sy}, x={sx}) lane {lane} row {sy - yb} of a {'rough' if rough else 'plain'} group, "
                           f"footprint (y0={p[1]}, x0={p[0]}): {', '.join(rel) or 'no merge'}")
    return f"({name} strips) " + ("; ".join(out) or "no source lands there")


def check_exact(got, ref, what, flow=None, geom=PIPE_GEOM):
    """Bit for bit: `got` (a CUDA tensor) == the fp64 value `ref` cast once to got's dtype. Names the first wrong element
    (frame, channel, row, column) and, given the flow, the merges of the sources that land on it."""
    want = torch.from_numpy(np.ascontiguousarray(ref)).to(got.dtype)
    g = got.detach().cpu()
    bad = ~((g == want) | (torch.isnan(g) & torch.isnan(want)))
    if bad.any():
        idx = _where(bad.numpy(), g.shape)
        raise AssertionError(f"{what}: {int(bad.sum())}/{g.numel()} elements differ from the exact value; first at "
                             f"(n, c, y, x) = {idx}: got {g[idx].item()!r} want {want[idx].item()!r}"
                             + ("" if flow is None else f"\n  merges there: {merges_at(flow, idx[0], idx[2], idx[3], geom)}"))


def check_ulps(got, ref, what, ulps=2, flow=None, geom=PIPE_GEOM):
    """Per element within `ulps` fp32 ulps of the fp64 value (1 ulp of a bf16 / fp16 output, which rounds once more)."""
    g = got.detach().cpu().double().numpy()
    tol = _ulp(ref, torch.float32) * ulps if got.dtype == torch.float32 else _ulp(ref, got.dtype)
    bad = ~(np.abs(g - ref) <= tol)
    if bad.any():
        idx = _where(bad, g.shape)
        raise AssertionError(f"{what}: {int(bad.sum())}/{g.size} elements off by more than {ulps} ulp; first at (n, c, y, x) "
                             f"= {idx}: got {g[idx]!r} want {ref[idx]!r}"
                             + ("" if flow is None else f"\n  merges there: {merges_at(flow, idx[0], idx[2], idx[3], geom)}"))


def _dev(a, dtype, layout=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(device="cuda", dtype=dtype)
    return t.contiguous(memory_format=layout) if layout is not None else t


def _follow_up(dcb, orc, shape):
    """One more ordinary sum splat through the same (kept-zero) workspace: exact again."""
    n, c, h, w = shape
    data, flow = dyadic_data(99, (n, c, h, w)), dyadic_flow(98, n, h, w, far=False)
    check_exact(dcb.softsplat(_dev(data, torch.float32), _dev(flow, torch.float32), None, "sum"), orc.splat_fwd(data, flow),
                "follow-up sum splat through the same workspace")


def run_family(dcb, orc, shape, mode, dtype=torch.float32, flow_dtype=None, layout=None, mask=False, seed=1, flow=None,
               geom=PIPE_GEOM):
    """One forward of the exact field through softsplat (or _splat_normalised with a mask factor), checked per element:
    sum and masked sum bit for bit, avg / linear within 2 ulps. Returns the output."""
    n, c, h, w = shape
    flow = dyadic_flow(seed, n, h, w) if flow is None else flow
    data = dyadic_data(seed + 1, shape)
    metric = dyadic_metric(seed + 2, n, h, w) if mode == "linear" else None
    m = np.random.default_rng(seed + 3).integers(0, 9, size=(n, 1, h, w)) / 8.0 if mask else None
    ref, _ = _orc_fwd(orc, data, flow, mode, metric, m)
    fdt = dtype if flow_dtype is None else flow_dtype
    ti, fl = _dev(data, dtype, layout), _dev(flow, fdt)
    me = None if metric is None else _dev(metric, dtype)
    what = f"{mode} {tuple(shape)} {dtype} flow {fdt}{' channels_last' if layout is not None else ''}{' (1 - mask)' if mask else ''}"
    if mode == "sum":
        out = dcb.softsplat(ti, fl, None, "sum")
    else:
        # the normalised modes with the zeroeps rule (an exact normaliser) and the optional mask factor: the entry behind
        # softsplat(..., "linear-zeroeps") and FeatureWarperSoftsplat ('avg-zeroeps' keeps the reference's quirk of
        # appending no channel, so avg is called here directly)
        ss = importlib.import_module(dcb.__name__ + ".softsplat")
        L = dcb._lib
        out = ss._splat_normalised(ti, fl, me, {"avg": L.MODE_AVG, "linear": L.MODE_LINEAR}[mode], L.EPS_ZERO,
                                   mask=None if m is None else _dev(m, dtype))
    torch.cuda.synchronize()
    if mode == "sum":
        check_exact(out, ref, what, flow, geom)
    else:                    # the mask factor is one more rounding: (1/d) * (1 - m), then the product with the sum
        check_ulps(out, ref, what, ulps=3 if mask else 2, flow=flow, geom=geom)
    return out


def raw_normaliser(dcb, orc, shape, mode, dtype=torch.float32, seed=1):
    """dcb_splat_fwd through the raw ABI with a normaliser descriptor: the saved normaliser (zeroeps) is exact."""
    L = dcb._lib
    lib = L.lib()
    n, c, h, w = shape
    flow, data = dyadic_flow(seed, n, h, w), dyadic_data(seed + 1, shape)
    metric = dyadic_metric(seed + 2, n, h, w) if mode == "linear" else None
    ref, ref_norm = _orc_fwd(orc, data, flow, mode, metric)
    ti, fl = _dev(data, dtype), _dev(flow, dtype)
    me = None if metric is None else _dev(metric, dtype)
    out = torch.empty_like(ti)
    norm = torch.empty((n, 1, h, w), dtype=torch.float64 if dtype == torch.float64 else torch.float32, device="cuda")
    md = {"avg": L.MODE_AVG, "linear": L.MODE_LINEAR}[mode]
    dt = L._DTYPES[dtype]
    need = lib.dcb_splat_fwd_workspace_bytes(n, c, h, w, dt, md, 0)
    ws = torch.zeros(max(need, 256), dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    L.check(lib.dcb_splat_fwd(L.desc(ti), L.desc(fl), L.desc(me), L.desc(out), L.desc(norm), None, ws.data_ptr(), ws.numel(),
                              md, L.EPS_ZERO, 0, st), "dcb_splat_fwd")
    torch.cuda.synchronize()
    check_exact(norm, ref_norm, f"{mode} saved normaliser {tuple(shape)} {dtype}")
    check_ulps(out, ref, f"{mode} raw ABI {tuple(shape)} {dtype}")


MODES = ["sum", "avg", "linear"]
PIPE = (PIPE_SHAPE[0], 3, PIPE_SHAPE[1], PIPE_SHAPE[2])


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the bit-exact matrix of forward families
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("opts", [{}, {"fwd_path": 1, "pipe_tail_percent": TAIL_PERCENT},
                                  {"fwd_path": 1, "pipe_group_bytes": 45 * 200 * 16}, {"fwd_path": 1, "pipe_ring_slots": 2,
                                                                                       "pipe_group_bytes": 45 * 200 * 16}],
                         ids=["default", "tail", "groups", "ring2"])
def test_pipeline_exact(dcb, orc, mode, opts):
    """The accumulator pipeline (C + 1 <= 4): one group, the single-pass tail strips, several ragged frame groups (one
    frame each), the two-slot ring. C = 1 and 3 (3 and 4 accumulated channels), C = 2 in sum mode."""
    geom = PIPE_TAIL_GEOM if "pipe_tail_percent" in opts else PIPE_GEOM
    with options(dcb, **opts):
        for c in ((1, 3) if mode != "sum" else (1, 2, 3)):
            run_family(dcb, orc, (PIPE[0], c, PIPE[2], PIPE[3]), mode, geom=geom)
        if mode != "sum":
            raw_normaliser(dcb, orc, PIPE, mode)
        _follow_up(dcb, orc, PIPE)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,flow_dtype", [(torch.bfloat16, torch.float32), (torch.bfloat16, torch.bfloat16),
                                              (torch.float16, torch.float32), (torch.float16, torch.float16)])
@pytest.mark.parametrize("family", ["pipe", "planar", "small"])
def test_half_storage_exact(dcb, orc, family, dtype, flow_dtype):
    """bf16 / fp16 storage, fp32 or same-dtype flow: one correctly rounded cast of the exact value (sum), 1 ulp (avg,
    linear)."""
    shape = {"pipe": PIPE, "planar": (2, 6, 45, 200), "small": (2, 3, 45, 90)}[family]
    for mode in MODES:
        run_family(dcb, orc, shape, mode, dtype, flow_dtype, geom=PLANAR_GEOM if family == "planar" else PIPE_GEOM)
    _follow_up(dcb, orc, shape)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_small_frame_exact(dcb, orc, mode):
    """The small-frame cluster kernel (default dispatch for H * W <= 8192, N <= 64, C + 1 <= 8)."""
    for shape in [(2, 3, 45, 90), (4, 7, 33, 70), (1, 1, 90, 37)]:
        run_family(dcb, orc, shape, mode)
    if mode != "sum":
        raw_normaliser(dcb, orc, (2, 3, 45, 90), mode)
    _follow_up(dcb, orc, (2, 3, 45, 90))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("one_launch", [0, 1])
def test_planar_exact(dcb, orc, mode, one_launch):
    """The planar channel-quad pipeline (C + 1 > 4 below the list threshold): C = 6, 9, 19 NCHW and C = 8 channels-last
    (one vector load per quad), with and without the single-launch kernel."""
    with options(dcb, planar_one_launch=one_launch, fwd_path=1):
        for shape, layout in [((2, 6, 45, 200), None), ((3, 9, 45, 70), None), ((1, 19, 29, 100), None),
                              ((2, 8, 45, 200), torch.channels_last)]:
            run_family(dcb, orc, shape, mode, layout=layout, geom=PLANAR_GEOM)
        if mode != "sum":
            raw_normaliser(dcb, orc, (2, 6, 45, 200), mode)
        _follow_up(dcb, orc, PIPE)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("nhwc", [1, 0])
def test_lists_exact(dcb, orc, mode, nhwc):
    """The per-target lists (C >= 16 at >= 16 MB): NCHW with C = 16, channels-last with C = 32 through the channels-last
    gather (lists_nhwc on) and the NCHW gather (off)."""
    with options(dcb, lists_nhwc=nhwc):
        L = dcb._lib
        for shape, layout in [((2, 16, 256, 512), None), ((1, 32, 256, 512), torch.channels_last)]:
            n, c, h, w = shape
            md = {"sum": L.MODE_SUM, "avg": L.MODE_AVG, "linear": L.MODE_LINEAR}[mode]
            assert L.fwd_is_scratch(n, c, h, w, L.DCB_F32, md)          # the list path
            run_family(dcb, orc, shape, mode, layout=layout, flow=dyadic_flow(5, n, h, w))
        _follow_up(dcb, orc, PIPE)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_owner_exact(dcb, orc, mode, dtype):
    """The target-tile owner kernels (fwd_path = 2; fp32 / bf16)."""
    with options(dcb, fwd_path=2):
        for c in (1, 3):
            run_family(dcb, orc, (PIPE[0], c, PIPE[2], PIPE[3]), mode, dtype)
        run_family(dcb, orc, (2, 3, 45, 90), mode, dtype)
        _follow_up(dcb, orc, PIPE)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_fp64_and_deterministic_exact(dcb, orc, mode):
    """fp64 tensors (the plain two-kernel path) and deterministic mode (sort-then-reduce) on the same fields."""
    for c in (3, 6):
        run_family(dcb, orc, (PIPE[0], c, PIPE[2], PIPE[3]), mode, torch.float64)
    with dcb.deterministic(True):
        for shape in [PIPE, (2, 3, 45, 90), (2, 6, 45, 200)]:
            run_family(dcb, orc, shape, mode)
    _follow_up(dcb, orc, PIPE)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["avg", "linear"])
@pytest.mark.parametrize("family", ["pipe", "small", "planar"])
def test_mask_factor_exact(dcb, orc, mode, family):
    """The (1 - mask) factor of FeatureWarperSoftsplat with a dyadic mask, fused into the normalise epilogue (the library
    takes a mask in the normalised modes only)."""
    shape = {"pipe": PIPE, "small": (2, 3, 45, 90), "planar": (2, 6, 45, 200)}[family]
    run_family(dcb, orc, shape, mode, mask=True, geom=PLANAR_GEOM if family == "planar" else PIPE_GEOM)
    _follow_up(dcb, orc, shape)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the sum-mode backward, exact
# ---------------------------------------------------------------------------------------------------------------------
BWD_NAMES = ("in", "flow")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(3, 1, 45, 200), (2, 3, 45, 90), (2, 19, 29, 70)])
def test_sum_backward_exact(dcb, orc, shape):
    """grad_in = sum of w * gout and grad_flow = sum of +-(1 - d or d) * v * gout are exact on the dyadic field with a
    dyadic upstream gradient: bit for bit against the fp64 oracle through autograd, for every gradient subset.
    The sum mode always takes the generic backward (csrc/splat_bwd.cu packed_bwd excludes it), so the packed path's options
    (bwd_flat, bwd_group_bytes) do not apply; the packed path's normalised-mode gradients divide by the normaliser and are
    not exact, and test_backward_paths_gpu.py covers them against the oracle."""
    n, c, h, w = shape
    flow = dyadic_flow(11, n, h, w)
    data, gout = dyadic_data(12, shape), dyadic_data(13, shape)
    t = {k: torch.from_numpy(v) for k, v in (("in", data), ("flow", flow))}
    for r in (1, 2):
        for want in itertools.combinations(BWD_NAMES, r):
            leaves = {k: t[k].clone().requires_grad_(k in want) for k in BWD_NAMES}
            orc.OracleSplatFunc.apply(leaves["in"], leaves["flow"]).backward(torch.from_numpy(gout))
            dev = {k: t[k].float().cuda().requires_grad_(k in want) for k in BWD_NAMES}
            out = dcb.softsplat(dev["in"], dev["flow"], None, "sum")
            out.backward(torch.from_numpy(gout).float().cuda())
            check_exact(out, orc.splat_fwd(data, flow), f"sum forward {shape}")
            for k in want:
                check_exact(dev[k].grad, leaves[k].grad.numpy(), f"sum backward grad {k} {shape} (asked for {want})")
            for k in BWD_NAMES:
                if k not in want:
                    assert dev[k].grad is None


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the recipe rider, checked through bit-equal masks
# ---------------------------------------------------------------------------------------------------------------------
def _check_image_side(got, ref, what, dtype):
    """fused / residual vs the fp64 oracle per element. Soft with the all-ones metric multiplies by e (inexact), so each
    piece is rounded once and the sums of <= ~10 positive pieces, the normaliser, the reciprocal, the fusion weights and
    the subtraction add a handful of fp32 roundings: 64 fp32 ulps of the element's magnitude (images are >= 0, nothing
    cancels before the residual). In bf16 the warped frames, the fused frame and the residual are each rounded to bf16
    (8 significant bits): 2^-6 of the magnitude."""
    g = got.detach().cpu().double().numpy()
    scale = np.abs(ref[0]) + np.abs(ref[1])            # |fused| + |value|: the residual's error is the fused one's
    tol = (2.0 ** -6 if dtype == torch.bfloat16 else 64 * 2.0 ** -24) * scale
    bad = ~(np.abs(g - ref[1]) <= tol)
    if bad.any():
        idx = _where(bad, g.shape)
        raise AssertionError(f"{what}: {int(bad.sum())}/{g.size} elements off; first at {idx}: got {g[idx]!r} want {ref[1][idx]!r}")


def _check_masks(got, ref, what, flow):
    g = got.detach().float().cpu()
    bad = g != ref.float()
    if bad.any():
        idx = _where(bad.numpy(), g.shape)
        raise AssertionError(f"{what}: {int(bad.sum())} mask entries differ from the oracle (no flip is allowed here); first at "
                             f"(n, 0, y, x) = {idx}: got {g[idx].item()} want {ref[idx].item()}\n"
                             f"  merges there: {merges_at(flow.numpy(), idx[0], idx[2], idx[3])}")


def _rider_inputs(dtype, c=3, swap=False):
    n, h, w = RIDER_SHAPE
    u = RIDER_U[dtype]
    flow1, flow2 = rider_flows(2, n, h, w, u)
    if swap:
        flow1, flow2 = flow2, flow1
    rng = np.random.default_rng(7)
    img1, img2, gt = (rng.integers(0, 9, size=(n, c, h, w)) / 8.0 for _ in range(3))
    # what the kernels read (1e9 is not a bf16 value), in fp64 for the oracle
    return [torch.from_numpy(a).to(dtype).double() for a in (img1, img2, flow1, flow2, gt)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("variant", ["dataset", "wrapper"])
@pytest.mark.parametrize("group_frames", [0, 1])
def test_recipe_rider_exact_masks(dcb, orc, variant, dtype, group_frames):
    """residual_conditioning on the accumulator pipeline (one or several frame groups): the rider pass's mask is bit-equal
    to the oracle's, and fused / residual within a few ulps per element."""
    n, h, w = RIDER_SHAPE
    img1, _, flow1, flow2, gt = _rider_inputs(dtype)
    with options(dcb, fwd_path=1, pipe_group_bytes=group_frames * h * w * 16):
        fused_r, res_r, of_r, ob_r = orc.residual_recipe(img1, flow1, flow2, gt, variant)
        dev = [t.to(device="cuda", dtype=dtype) for t in (img1, flow1, flow2, gt)]
        fused, res, of, ob = dcb.residual_conditioning(*dev, variant, return_masks=True)
        torch.cuda.synchronize()
        what = f"recipe {variant} {dtype} groups of {group_frames or n}"
        _check_masks(ob, ob_r, what + ": rider mask compute_mask(flow2, flow1)", flow1)
        _check_masks(of, of_r, what + ": mask compute_mask(flow1, flow2)", flow2)
        _check_image_side(fused, (fused_r.numpy(), fused_r.numpy()), what + " fused", dtype)
        _check_image_side(res, (fused_r.numpy(), res_r.numpy()), what + " residual", dtype)
        _follow_up(dcb, orc, (n, 3, h, w))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("swap", [False, True], ids=["rider_pass_B", "rider_pass_A"])
def test_bidir_rider_exact_masks(dcb, orc, dtype, swap):
    """residual_conditioning_bidir: pass A carries flow1 on flow2, pass B flow2 on flow1; swapping the flows puts the
    constant rider in either pass. Both masks bit-equal to the oracle's."""
    n, h, w = RIDER_SHAPE
    img1, img2, flow1, flow2, gt = _rider_inputs(dtype, swap=swap)
    with options(dcb, fwd_path=1, pipe_group_bytes=h * w * 16):
        ones = torch.ones_like(flow1[:, :1])
        w1, w2 = orc.softsplat(img1, flow1, ones, "soft"), orc.softsplat(img2, flow2, ones, "soft")
        of_r, ob_r = orc.compute_mask(flow1, flow2), orc.compute_mask(flow2, flow1)
        fused_r = orc.soft_fuse(w1, w2, 1 - of_r, 1 - ob_r)
        dev = [t.to(device="cuda", dtype=dtype) for t in (img1, img2, flow1, flow2, gt)]
        fused, res, of, ob = dcb.residual_conditioning_bidir(*dev, return_masks=True)
        torch.cuda.synchronize()
        what = f"bidir {dtype} {'flows swapped' if swap else ''}"
        _check_masks(of, of_r, what + ": pass A mask compute_mask(flow1, flow2)", flow2)
        _check_masks(ob, ob_r, what + ": pass B mask compute_mask(flow2, flow1)", flow1)
        _check_image_side(fused, (fused_r.numpy(), fused_r.numpy()), what + " fused", dtype)
        _check_image_side(res, (fused_r.numpy(), (gt - fused_r).numpy()), what + " residual", dtype)
        _follow_up(dcb, orc, (n, 3, h, w))
