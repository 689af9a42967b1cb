"""Focal loss, Gaussian target splat and Reg*Loss (csrc/focal.cu, DESIGN rows A13-A16) on every code path.

Each of these losses writes, in its forward pass, the gradient the trainer back-propagates.  A wrong gradient
crashes nothing and only makes training worse, so every test here checks every gradient element, not only the
loss value.  References:
  * losses_np.neg_loss: fp32 element terms in the reference's operation order, float64 sums;
  * losses_np.neg_loss_grad / neg_loss_grad_logits: float64 (the logits form takes torch's CUDA sigmoid, which
    the library reproduces bit for bit, test_logits_gpu.py);
  * image_np.splat_objects: draw_umich_gaussian, clipped windows included;
  * float64 torch autograd on the CPU of the reference's Reg*Loss formulas.
Bars: loss values rtol 1e-5 (SURVEY 8d); targets bit for bit (the table and the direct path both evaluate
draw_umich_gaussian's float64 expression and round once to fp32, DESIGN 4.3); gradients
|g - ref| <= 1e-5 |ref| + 1e-6 max|ref| per element: the two terms of each branch of the focal gradient have
the same sign, so nothing cancels."""
import functools
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import image_np, losses_np

pytestmark = pytest.mark.gpu

F32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LO, HI = F32(1e-4), F32(1 - 1e-4)          # the clamp of _sigmoid (models/utils.py:8-10)


# ------------------------------------------------------------------ helpers
def cuda(*arrs):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs]


def _input(v, offset=0):
    """v on the device as a differentiable view `offset` floats into its buffer.  offset=1 leaves it contiguous
    (no copy on the way in) but not 16-byte aligned, so the kernels run their scalar loops."""
    buf = torch.zeros(v.size + offset, device="cuda")
    buf[offset:] = torch.from_numpy(np.ascontiguousarray(v, F32).ravel()).cuda()
    buf.requires_grad_(True)
    x = buf[offset:].view(v.shape)
    assert (x.data_ptr() % 16 == 0) == (offset % 4 == 0)
    return buf, x


def _grad(buf, shape, offset=0):
    assert not buf.grad[:offset].any(), "gradient written in front of the input"
    return buf.grad[offset:].view(shape)


def assert_loss(got, want, what=""):
    np.testing.assert_allclose(float(got), float(want), rtol=1e-5, err_msg=what)


def assert_grad(got, want, what=""):
    if torch.is_tensor(got):
        got = got.detach().cpu().numpy()
    want = np.asarray(want, np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    err = np.abs(got.astype(np.float64) - want)
    bound = 1e-5 * np.abs(want) + 1e-6 * np.abs(want).max()
    bad = err > bound
    if bad.any():
        i = np.unravel_index(np.argmax(err - bound), want.shape)
        raise AssertionError("%s: %d of %d gradient elements off; worst at %s: got %r, want %r"
                             % (what, int(bad.sum()), bad.size, tuple(int(k) for k in i), float(got[i]), want[i]))


def assert_targets_equal(got, want, what=""):
    bad = np.argwhere(got != want)
    assert not len(bad), "%s: %d target values differ, first (b, c, y, x, got, want): %s" % (
        what, len(bad), [(*map(int, k), float(got[tuple(k)]), float(want[tuple(k)])) for k in bad[:8]])


def focal_ref(v, gt, logits):
    """Oracle (loss, gradient) for the values the kernel reads: probabilities, or logits whose sigmoid is
    torch's CUDA sigmoid."""
    if not logits:
        return losses_np.neg_loss(v, gt)[0], losses_np.neg_loss_grad(v, gt)
    s32 = torch.sigmoid(torch.from_numpy(np.ascontiguousarray(v)).cuda()).cpu().numpy()
    return losses_np.neg_loss(np.clip(s32, LO, HI), gt)[0], losses_np.neg_loss_grad_logits(s32, gt)


def dense_loss(x, gt, logits):
    from centernet_b200 import losses as L
    return L._neg_loss_from_logits(x, gt) if logits else L.FocalLoss()(x, gt)


def objects(rng, B, M, C, H, W):
    """Object lists as datasets/sample/ctdet.py:99-117 writes them: integer centres, and radii
    max(0, int(gaussian_radius(ceil(h), ceil(w)))) of boxes up to the size of the map."""
    cls = rng.integers(0, C, (B, M), dtype=np.int32)
    cx = rng.integers(0, W, (B, M), dtype=np.int32)
    cy = rng.integers(0, H, (B, M), dtype=np.int32)
    bh, bw = rng.uniform(0.5, H, (B, M)), rng.uniform(0.5, W, (B, M))
    rad = np.array([[max(0, int(image_np.gaussian_radius((math.ceil(h), math.ceil(w))))) for h, w in zip(rh, rw)]
                    for rh, rw in zip(bh, bw)], np.int32)
    return cls, cx, cy, rad, np.ones((B, M), np.uint8)


def dense_inputs(shape, seed):
    """Logits with the head's bias prior (tails beyond the clamp) and a target with exact 0s, 1s and values
    spread over (0, 1)."""
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal(shape) * 3 - 2.19).astype(F32)
    gt = (rng.random(shape) ** 4).astype(F32)
    gt[rng.random(shape) < 0.1] = 0
    gt[rng.random(shape) < 0.01] = 1
    gt.flat[0] = 1
    return x, gt


def pred_values(x, logits):
    return x if logits else losses_np.sigmoid_clamped(x)


@functools.lru_cache(maxsize=None)
def training_case():
    """BASELINE's training geometry: 8 x 80 x 128 x 128, 128 objects per image."""
    B, C, H, W, M = 8, 80, 128, 128, 128
    rng = np.random.default_rng(2026)
    objs = objects(rng, B, M, C, H, W)
    gt = image_np.splat_objects(*objs, C, H, W)
    x = (rng.standard_normal((B, C, H, W)) * 3 - 2.19).astype(F32)
    return objs, gt, x


def check_dense(x, gt, logits, offset=0, what=""):
    v = pred_values(x, logits)
    buf, p = _input(v, offset)
    _, g = _input(gt, offset)
    loss = dense_loss(p, g.detach(), logits)
    loss.backward()
    got = _grad(buf, v.shape, offset).cpu().numpy()
    want_loss, want_grad = focal_ref(v, gt, logits)
    assert_loss(loss.item(), want_loss, what)
    assert_grad(got, want_grad, what)
    return got, want_grad


def check_splat(objs, C, H, W, x=None, logits=False, offset=0, seed=0, what=""):
    """splat_gaussian bit for bit against draw_umich_gaussian.  FocalSplatLoss against the focal oracle on that
    target, and its gradient bit for bit against the dense kernel's on the oracle's target: both run the same
    per-element arithmetic, so a difference there is a difference in the target the splat loss rebuilt."""
    from centernet_b200 import losses as L
    B = objs[0].shape[0]
    want = image_np.splat_objects(*objs, C, H, W)
    d_objs = cuda(*objs)
    assert_targets_equal(L.splat_gaussian(*d_objs, C, H, W).cpu().numpy(), want, what + " splat_gaussian")
    if x is None:
        x = (np.random.default_rng(seed).standard_normal((B, C, H, W)) * 3 - 2.19).astype(F32)
    v = pred_values(x, logits)
    buf, p = _input(v, offset)
    loss = L.FocalSplatLoss(from_logits=logits)(p, *d_objs)
    loss.backward()
    got = _grad(buf, v.shape, offset)
    want_loss, want_grad = focal_ref(v, want, logits)
    assert_loss(loss.item(), want_loss, what)
    assert_grad(got, want_grad, what)
    q = cuda(v)[0].requires_grad_(True)
    dense_loss(q, cuda(want)[0], logits).backward()
    assert torch.equal(got, q.grad), what + ": FocalSplatLoss's gradient differs from the dense kernel's on the " \
                                            "oracle target (the rebuilt target is not bit-identical)"
    return loss.item()


# ------------------------------------------------------------------ dense FocalLoss / _neg_loss_from_logits
@pytest.mark.parametrize("logits", [False, True], ids=["prob", "logits"])
def test_dense_training_size(logits):
    """Eight CTAs per SM: num_pos normalisation across CTAs, the last-CTA finish, every gradient element."""
    objs, gt, x = training_case()
    assert (objs[3] >= 27).sum() >= 16
    got, want = check_dense(x, gt, logits, what="training size")
    if logits:
        assert (want == 0).any() and not got[want == 0].any()     # logits outside the clamp


@pytest.mark.parametrize("shape", [(3, 5, 7, 9), (2, 3, 5, 7), (1, 1, 1, 3)])
@pytest.mark.parametrize("logits", [False, True], ids=["prob", "logits"])
def test_dense_scalar_tail(shape, logits):
    """n % 4 != 0: the last elements go through the scalar tail after the float4 loop (all of them for n < 4)."""
    x, gt = dense_inputs(shape, 11)
    check_dense(x, gt, logits, what=str(shape))


@pytest.mark.parametrize("logits", [False, True], ids=["prob", "logits"])
def test_dense_misaligned(logits):
    """pred and gt one float into their buffers: contiguous, so not copied, and handled by the non-float4 loop."""
    x, gt = dense_inputs((4, 16, 64, 64), 12)
    check_dense(x, gt, logits, offset=1, what="misaligned")


def test_logits_outside_clamp_have_zero_gradient():
    """clamp's backward passes the gradient only inside [1e-4, 1-1e-4], bounds included."""
    shape = (2, 8, 64, 64)
    x, gt = dense_inputs(shape, 13)
    rng = np.random.default_rng(14)
    far = rng.random(shape) < 0.4
    x[far] = (np.sign(rng.standard_normal(shape)) * (9.3 + 20 * rng.random(shape)))[far].astype(F32)
    # every float within 4096 ulp of the two logits where the sigmoid crosses the bounds
    sweep = [(np.array([e], F32).view(np.int32) + np.arange(-4096, 4096, dtype=np.int32)).view(F32)
             for e in (-9.21024, 9.21024)]
    sweep = np.concatenate(sweep)
    x.reshape(-1)[1:1 + sweep.size] = sweep
    s32 = torch.sigmoid(torch.from_numpy(x).cuda()).cpu().numpy()
    assert (s32 == HI).any() and (s32 < LO).any() and (s32 > HI).any()
    got, want = check_dense(x, gt, True, what="saturated logits")
    assert (got[np.abs(x) > 9.3] == 0).all()
    assert not got[want == 0].any()


@pytest.mark.parametrize("logits", [False, True], ids=["prob", "logits"])
def test_dense_no_positive_multi_cta(logits):
    """num_pos = 0: the loss is -neg_sum and the gradient is not normalised."""
    x, gt = dense_inputs((2, 80, 128, 128), 15)
    gt = np.minimum(gt, F32(0.5))
    assert not (gt == 1).any()
    check_dense(x, gt, logits, what="no positive")


@pytest.mark.parametrize("logits", [False, True], ids=["prob", "logits"])
def test_dense_target_above_one_contributes_nothing(logits):
    """gt > 1 is neither positive (== 1) nor negative (< 1) in _neg_loss: no loss, no gradient."""
    x, gt = dense_inputs((2, 6, 32, 36), 16)
    rng = np.random.default_rng(17)
    above = rng.random(gt.shape) < 0.2
    gt[above] = (1 + 2 * rng.random(gt.shape))[above].astype(F32)
    gt.reshape(-1)[1:4] = [np.nextafter(F32(1), F32(2)), F32(2), F32(1)]
    above = gt > 1
    got, _ = check_dense(x, gt, logits, what="gt > 1")
    assert (got[above] == 0).all()


def test_focal_backward_scales_accumulates_and_keeps_layout():
    """backward with grad_out != 1, one pred feeding two losses, and a non-contiguous (permuted) pred."""
    from centernet_b200 import losses as L
    B, C, H, W, M = 2, 6, 32, 40, 12
    x, gt = dense_inputs((B, C, H, W), 18)
    objs = objects(np.random.default_rng(19), B, M, C, H, W)
    gs = image_np.splat_objects(*objs, C, H, W)
    d_gt, = cuda(gt)
    d_objs = cuda(*objs)
    for logits in (False, True):
        v = pred_values(x, logits)
        _, dense_grad = focal_ref(v, gt, logits)
        _, splat_grad = focal_ref(v, gs, logits)
        p = cuda(v)[0].requires_grad_(True)
        (0.37 * dense_loss(p, d_gt, logits)).backward()
        assert_grad(p.grad, 0.37 * dense_grad, "0.37 * FocalLoss, logits=%s" % logits)
        p = cuda(v)[0].requires_grad_(True)
        (0.37 * L.FocalSplatLoss(from_logits=logits)(p, *d_objs)).backward()
        assert_grad(p.grad, 0.37 * splat_grad, "0.37 * FocalSplatLoss, logits=%s" % logits)
        p = cuda(v)[0].requires_grad_(True)
        (dense_loss(p, d_gt, logits) - 2.5 * L.FocalSplatLoss(from_logits=logits)(p, *d_objs)).backward()
        assert_grad(p.grad, dense_grad - 2.5 * splat_grad, "two losses, logits=%s" % logits)
        # a channels-last leaf seen as [B, C, H, W]: the gradient lands on the right elements, in its layout
        p = cuda(v.transpose(0, 2, 3, 1))[0].permute(0, 3, 1, 2).requires_grad_(True)
        assert not p.is_contiguous()
        keep = p.detach().clone()
        dense_loss(p, d_gt, logits).backward()
        assert torch.equal(p.detach(), keep)
        assert p.grad.stride() == p.stride()
        assert_grad(p.grad, dense_grad, "permuted pred, logits=%s" % logits)


# ------------------------------------------------------------------ splat_gaussian / FocalSplatLoss
@pytest.mark.parametrize("W", [160, 157], ids=["float4", "scalar"])
def test_splat_radius_sweep_bit_exact(W):
    """r = 0..80, one object per plane, centred so that a full quadrant of the window of every radius that has a
    table lies inside the map: every table entry a pixel can read is checked.  r >= 56 does not fit the
    shared-memory table and takes the direct path."""
    from centernet_b200 import losses as L
    R = 80
    H, C = 2 * R + 1, R + 1
    r = np.arange(C, dtype=np.int32)[None]
    objs = (r.copy(), np.full_like(r, W // 2), np.full_like(r, R), r.copy(), np.ones(r.shape, np.uint8))
    want = image_np.splat_objects(*objs, C, H, W)
    got = L.splat_gaussian(*cuda(*objs), C, H, W).cpu().numpy()
    bad = np.argwhere(got != want)
    pairs = sorted({(int(c), int((xx - W // 2) ** 2 + (yy - R) ** 2)) for _, c, yy, xx in bad})
    assert not pairs, "targets differ from draw_umich_gaussian at (r, d2): %s" % pairs[:20]
    check_splat(objs, C, H, W, seed=20, what="radius sweep")


@pytest.mark.parametrize("W", [128, 125], ids=["float4", "scalar"])
def test_splat_table_overflow_by_accumulation(W):
    """Four overlapping r = 34 objects of one class (2313 table floats each, 6144 in all): the third and fourth
    take the direct path, and their values meet the tabled ones inside fmaxf.  Small objects after them still
    get tables; a single r = 60 object overflows on its own."""
    H, C = 128, 3
    rows = [(0, 40, 40, 34), (0, 52, 46, 34), (0, 45, 57, 34), (0, 61, 50, 34), (0, 50, 50, 3), (0, 90, 100, 10),
            (1, 64, 64, 60), (1, 70, 60, 5), (2, 10, 120, 34), (2, 20, 110, 34), (2, 30, 100, 34), (2, 40, 90, 34),
            (2, 50, 80, 34), (2, 25, 105, 0)]
    c, x, y, r = (np.array([[t[k] for t in rows]], np.int32) for k in range(4))
    objs = (c, x, y, r, np.ones(c.shape, np.uint8))
    for logits in (False, True):
        check_splat(objs, C, H, W, logits=logits, seed=21, what="overflow W=%d logits=%s" % (W, logits))


@pytest.mark.parametrize("W", [44, 43], ids=["float4", "scalar"])
def test_splat_clipped_windows(W):
    """Centres on the corners and edges with radii beyond the border: draw_umich_gaussian's clipped windows."""
    H, C = 37, 4
    pts = [(0, 0), (W - 1, 0), (0, H - 1), (W - 1, H - 1), (W // 2, 0), (0, H // 2), (W - 1, H // 2),
           (W // 2, H - 1), (1, 1), (W - 2, H - 2)]
    radii = [5, 12, 40, 7, 20, 3, 60, 9, 18, 25]
    c = np.array([[k % C for k in range(len(pts))] * 2], np.int32)
    x = np.array([[p[0] for p in pts] * 2], np.int32)
    y = np.array([[p[1] for p in pts] * 2], np.int32)
    r = np.array([radii + radii[::-1]], np.int32)
    objs = (c, x, y, r, np.ones(c.shape, np.uint8))
    for logits in (False, True):
        check_splat(objs, C, H, W, logits=logits, seed=22, what="clipped W=%d logits=%s" % (W, logits))


@pytest.mark.parametrize("W", [48, 45], ids=["float4", "scalar"])
def test_splat_duplicates_overlaps_and_invalid(W):
    """One positive per distinct valid (cls, cx, cy): a repeated centre counts once and its target is the max of
    the two Gaussians; the same centre in two classes counts twice; invalid objects draw and count nothing;
    an image may have no valid object, and a batch none at all (num_pos = 0, un-normalised gradient)."""
    from centernet_b200 import losses as L
    H, C, M = 40, 6, 8
    cls = np.zeros((3, M), np.int32); cx = np.zeros((3, M), np.int32); cy = np.zeros((3, M), np.int32)
    rad = np.zeros((3, M), np.int32); val = np.zeros((3, M), np.uint8)

    def put(b, m, c, x, y, r, v=1):
        cls[b, m], cx[b, m], cy[b, m], rad[b, m], val[b, m] = c, x, y, r, v

    put(0, 0, 2, 10, 12, 3); put(0, 1, 2, 10, 12, 9); put(0, 2, 5, 10, 12, 4)      # same centre: twice, two classes
    put(0, 3, 2, 14, 15, 6); put(0, 4, 2, 30, 20, 7, v=0); put(0, 5, 4, 20, 30, 0)  # overlap; invalid; r = 0
    put(0, 6, 2, 10, 12, 9); put(0, 7, 5, 11, 12, 4)                                 # exact duplicate; neighbour
    for m in range(M):                                                               # image 1: nothing valid
        put(1, m, m % C, 3 * m, 2 * m, m + 2, v=0)
    put(2, 0, 1, 0, 0, 8); put(2, 1, 1, 0, 0, 8); put(2, 2, 1, 0, 0, 2); put(2, 3, 1, 0, 0, 5, v=0)
    put(2, 4, 0, W - 1, H - 1, 11); put(2, 5, 3, 7, 7, 1, v=0)
    objs = (cls, cx, cy, rad, val)
    hm = image_np.splat_objects(*objs, C, H, W)
    assert (hm == 1).sum() == 5 + 2
    assert not hm[1].any()
    for logits in (False, True):
        check_splat(objs, C, H, W, logits=logits, seed=23, what="duplicates W=%d logits=%s" % (W, logits))
    # no valid object anywhere: loss = -neg_sum of an all-zero target
    none = (cls, cx, cy, rad, np.zeros_like(val))
    for logits in (False, True):
        check_splat(none, C, H, W, logits=logits, seed=24, what="no object W=%d logits=%s" % (W, logits))
    assert not L.splat_gaussian(*cuda(*none), C, H, W).any()


@pytest.mark.parametrize("H,W", [(6, 1028), (5, 1030), (1, 64), (1, 61)])
def test_splat_wide_and_thin_planes(H, W):
    """W = 1028: 257 float4 per row, more than the 256 threads of a CTA, so a thread's row never advances by a
    whole row per step.  W = 1030 and W = 61: scalar path.  H = 1: windows clipped to a single row."""
    rng = np.random.default_rng(25 + W)
    B, C, M = 2, 3, 24
    cls = rng.integers(0, C, (B, M), dtype=np.int32)
    cx = rng.integers(0, W, (B, M), dtype=np.int32)
    cy = rng.integers(0, H, (B, M), dtype=np.int32)
    rad = rng.integers(0, 40, (B, M), dtype=np.int32)
    cx[0, :4] = [0, W - 1, min(1020, W - 1), min(1024, W - 1)]
    objs = (cls, cx, cy, rad, np.ones((B, M), np.uint8))
    for logits in (False, True):
        check_splat(objs, C, H, W, logits=logits, seed=26, what="H=%d W=%d logits=%s" % (H, W, logits))


@pytest.mark.parametrize("logits", [False, True], ids=["prob", "logits"])
def test_focal_splat_training_size(logits):
    """FocalSplatLoss(from_logits) at 8 x 80 x 128 x 128 with 128 objects per image against the dense oracle
    built on splat_objects."""
    objs, gt, x = training_case()
    check_splat(objs, 80, 128, 128, x=x, logits=logits, what="training size")


@pytest.mark.parametrize("logits", [False, True], ids=["prob", "logits"])
def test_focal_splat_misaligned_pred(logits):
    """pred one float into its buffer: W % 4 == 0 but the loss takes the scalar path."""
    B, C, H, W, M = 2, 8, 64, 64, 40
    objs = objects(np.random.default_rng(27), B, M, C, H, W)
    objs[3][0, :4] = 34                                   # four r = 34 objects: some past the table
    check_splat(objs, C, H, W, logits=logits, offset=1, seed=28, what="misaligned pred")


# ------------------------------------------------------------------ row bands (CNB_FOCAL_PARTS)
BAND_W = (128, 125)


def band_inputs():
    """H = 128 split in 5 bands starts rows 0, 25, 51, 76, 102: uneven bands, and objects straddling each edge."""
    rng = np.random.default_rng(29)
    B, C, H, M = 2, 4, 128, 40
    case = {}
    for W in BAND_W:
        cls = rng.integers(0, C, (B, M), dtype=np.int32)
        cx = rng.integers(0, W, (B, M), dtype=np.int32)
        cy = rng.integers(0, H, (B, M), dtype=np.int32)
        rad = rng.integers(0, 30, (B, M), dtype=np.int32)
        edges = [0, 24, 25, 50, 51, 75, 76, 101, 102, 127]
        cy[:, :len(edges)] = edges
        rad[:, :len(edges)] = [3, 1, 30, 12, 0, 26, 2, 40, 25, 9]
        case.update({"cls%d" % W: cls, "cx%d" % W: cx, "cy%d" % W: cy, "rad%d" % W: rad,
                     "val%d" % W: np.ones((B, M), np.uint8),
                     "x%d" % W: (rng.standard_normal((B, C, H, W)) * 3 - 2.19).astype(F32)})
    return case


def band_outputs(case):
    """splat_gaussian and FocalSplatLoss (both forms) of band_inputs(), as numpy arrays."""
    from centernet_b200 import losses as L
    out = {}
    for W in BAND_W:
        objs = cuda(*(case[k + str(W)] for k in ("cls", "cx", "cy", "rad", "val")))
        x = case["x%d" % W]
        C, H = x.shape[1], x.shape[2]
        out["hm%d" % W] = L.splat_gaussian(*objs, C, H, W).cpu().numpy()
        for logits in (0, 1):
            p = cuda(pred_values(x, logits))[0].requires_grad_(True)
            loss = L.FocalSplatLoss(from_logits=bool(logits))(p, *objs)
            loss.backward()
            out["loss%d_%d" % (W, logits)] = np.float32(loss.item())
            out["grad%d_%d" % (W, logits)] = p.grad.cpu().numpy()
    return out


def _band_main(inp, outp):
    z = np.load(inp)
    np.savez(outp, **band_outputs({k: z[k] for k in z.files}))


def test_row_bands_match_whole_planes(tmp_path):
    """CNB_FOCAL_PARTS=5 (read once per process, so in a child process): targets and gradients bit for bit equal
    to the whole-plane run, loss within rtol 1e-5."""
    case = band_inputs()
    np.savez(tmp_path / "in.npz", **case)
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_focal_splat_gpu as t; t._band_main(%r, %r)"
            % (ROOT, os.path.dirname(os.path.abspath(__file__)), str(tmp_path / "in.npz"), str(tmp_path / "out.npz")))
    env = dict(os.environ, CNB_FOCAL_PARTS="5")
    r = subprocess.run([sys.executable] + subprocess._args_from_interpreter_flags() + ["-c", code], env=env,
                       cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    z = np.load(tmp_path / "out.npz")
    banded = {k: z[k] for k in z.files}
    whole = band_outputs(case)
    assert sorted(banded) == sorted(whole)
    for W in BAND_W:
        objs = [case[k + str(W)] for k in ("cls", "cx", "cy", "rad", "val")]
        C, H = case["x%d" % W].shape[1:3]
        assert_targets_equal(whole["hm%d" % W], image_np.splat_objects(*objs, C, H, W), "whole planes W=%d" % W)
        assert_targets_equal(banded["hm%d" % W], whole["hm%d" % W], "5 bands W=%d" % W)
        for logits in (0, 1):
            k = "%d_%d" % (W, logits)
            np.testing.assert_array_equal(banded["grad" + k], whole["grad" + k], err_msg="gradient " + k)
            np.testing.assert_allclose(banded["loss" + k], whole["loss" + k], rtol=1e-5, err_msg="loss " + k)


# ------------------------------------------------------------------ Reg*Loss
REG_MODES = [("RegL1Loss", 0), ("RegLoss", 1), ("NormRegL1Loss", 2), ("RegWeightedL1Loss", 3)]


def reg_inputs(B, M, D, H, W, mode, seed):
    """Rows as the datasets write them: live objects first, then padding (ind = 0, mask 0, target 0).  Some
    live rows repeat the index of an earlier live row (two objects on one output pixel)."""
    rng = np.random.default_rng(seed)
    output = (rng.standard_normal((B, D, H, W)) * 2).astype(F32)
    nlive = rng.integers(0, M + 1, B)
    nlive[0], nlive[1] = M, 0
    ind = np.zeros((B, M), np.int64)
    mask = np.zeros((B, M), np.uint8)
    for b in range(B):
        k = int(nlive[b])
        ind[b, :k] = rng.choice(H * W, k, replace=False)
        mask[b, :k] = 1
        for i in range(1, k):
            if rng.random() < 0.15:
                ind[b, i] = ind[b, rng.integers(0, i)]
    gathered = output.reshape(B, D, H * W).transpose(0, 2, 1)[np.arange(B)[:, None], ind]      # [B, M, D]
    if mode == 2:      # NormRegL1Loss: positive sizes
        target = rng.uniform(0.5, 40, (B, M, D)).astype(F32)
    else:              # around the prediction: |diff| on both sides of smooth-L1's 1
        target = (gathered + rng.standard_normal((B, M, D)) * 1.5).astype(F32)
    target *= mask[:, :, None]
    if mode == 3:      # float weights with zeros, zero on padding rows
        w = rng.random((B, M, D)).astype(F32)
        w[rng.random((B, M, D)) < 0.3] = 0
        mask = (w * mask[:, :, None]).astype(F32)
    return output, mask, ind, target


def reg_ref(output, mask, ind, target, mode, scale):
    """Float64 autograd of models/losses.py:97-175 on the CPU.  Returns (loss, d(scale * loss)/d output)."""
    o = torch.from_numpy(output).double().requires_grad_(True)
    B, D = o.shape[:2]
    ind = torch.from_numpy(ind)
    mask = torch.from_numpy(mask).double()
    t = torch.from_numpy(target).double()
    pred = o.view(B, D, -1).permute(0, 2, 1).gather(1, ind.unsqueeze(2).expand(B, ind.size(1), D))
    if mode == 1:
        m = mask.unsqueeze(2).expand_as(pred)
        loss = F.smooth_l1_loss(pred * m, t * m, reduction="sum") / (mask.sum() + 1e-4)
    else:
        m = mask if mode == 3 else mask.unsqueeze(2).expand_as(pred)
        if mode == 2:
            pred = pred / (t + 1e-4)
            t = t * 0 + 1
        loss = F.l1_loss(pred * m, t * m, reduction="sum") / (m.sum() + 1e-4)
    (scale * loss).backward()
    return loss.item(), o.grad.numpy()


@pytest.mark.parametrize("name,mode", REG_MODES, ids=[n for n, _ in REG_MODES])
@pytest.mark.parametrize("B,M,D", [(32, 128, 2), (16, 32, 34)], ids=["ctdet", "hps"])
def test_reg_loss(B, M, D, name, mode):
    """ctdet's wh / reg geometry and multi_pose's hps (D = 34): B*M*D > 1024, so every thread of the one CTA
    loops; duplicated live indices add their gradients; backward of 0.37 * loss."""
    from centernet_b200 import losses as L
    H = W = 128
    output, mask, ind, target = reg_inputs(B, M, D, H, W, mode, 30 + mode + D)
    want_loss, want_grad = reg_ref(output, mask, ind, target, mode, 0.37)
    o = cuda(output)[0].requires_grad_(True)
    loss = getattr(L, name)()(o, *cuda(mask, ind, target))
    (0.37 * loss).backward()
    assert_loss(loss.item(), want_loss, name)
    assert_grad(o.grad, want_grad, name)
