"""GPU parity for multi_pose_decode (A6), edge aggregation (A7), focal loss + target splat
(A13-A15) and the Reg*Loss family (A16): goldens from the reference + numpy-oracle sweeps."""
import numpy as np
import pytest
import torch

from helpers import assert_dets_equal, golden
from oracle import decode_np as O
from oracle import image_np, losses_np

pytestmark = pytest.mark.gpu
TOL = 1e-4


def dev(*arrs):
    return [None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs]


def rnd(shape, seed, scale=1.0, normal=False):
    g = torch.Generator().manual_seed(seed)
    t = torch.randn(*shape, generator=g) if normal else torch.rand(*shape, generator=g)
    return (t * scale).numpy()


def noise(B, C, H, W, seed, bias=2.19):
    g = torch.Generator().manual_seed(seed)
    return torch.sigmoid(torch.randn(B, C, H, W, generator=g) - bias).numpy()


# ------------------------------------------------------------------ multi_pose
def test_golden_multi_pose():
    from centernet_b200 import decode as D
    g = golden("multi_pose")
    K = int(g["K"])
    heat, wh, kps, reg, hm_hp, off = dev(g["heat"], g["wh"], g["kps"], g["reg"], g["hm_hp"], g["hp_offset"])
    got = D.multi_pose_decode(heat, wh, kps, reg=reg, hm_hp=hm_hp, hp_offset=off, K=K).cpu().numpy()
    assert_dets_equal(g["dets"], got, atol=TOL, what="multi_pose")
    got = D.multi_pose_decode(heat, wh, kps, reg=None, hm_hp=hm_hp, hp_offset=None, K=K).cpu().numpy()
    assert_dets_equal(g["dets_nooff"], got, atol=TOL, what="multi_pose_nooff")
    got = D.multi_pose_decode(heat, wh, kps, reg=reg, K=K).cpu().numpy()
    assert_dets_equal(g["dets_nohp"], got, atol=TOL, what="multi_pose_nohp")


@pytest.mark.parametrize("B,H,W,K", [(2, 128, 128, 100), (3, 40, 56, 32)])
def test_multi_pose_vs_oracle(B, H, W, K):
    from centernet_b200 import decode as D
    J = 17
    heat = noise(B, 1, H, W, 3)
    wh = rnd((B, 2, H, W), 4, 30.0); kps = rnd((B, 2 * J, H, W), 5, 8.0, normal=True)
    reg = rnd((B, 2, H, W), 6); hm_hp = noise(B, J, H, W, 7, bias=1.0); off = rnd((B, 2, H, W), 8)
    want = O.multi_pose_decode(heat, wh, kps, reg, hm_hp, off, K=K)
    got = D.multi_pose_decode(*dev(heat, wh, kps, reg, hm_hp, off), K=K).cpu().numpy()
    assert got.shape == (B, K, 40)
    np.testing.assert_array_equal(got[..., 4], want[..., 4])
    np.testing.assert_array_equal(got[..., -1], want[..., -1])
    np.testing.assert_allclose(got, want, rtol=0, atol=TOL)


# ------------------------------------------------------------------ edge aggregation (bit-exact: sequential fp32 sums)
def test_golden_aggregate():
    from centernet_b200 import decode as D
    g = golden("aggregate")
    heat, = dev(g["heat"])
    for name, fn in (("left", D._left_aggregate), ("right", D._right_aggregate), ("top", D._top_aggregate),
                     ("bottom", D._bottom_aggregate)):
        np.testing.assert_array_equal(fn(heat).cpu().numpy(), g[name], err_msg=name)
    np.testing.assert_array_equal(D._h_aggregate(heat, 0.1).cpu().numpy(), g["h"])
    np.testing.assert_array_equal(D._v_aggregate(heat, 0.1).cpu().numpy(), g["v"])


@pytest.mark.parametrize("B,C,H,W", [(2, 80, 128, 128), (1, 3, 70, 300), (2, 2, 5, 7), (1, 2, 33, 516), (1, 1, 600, 36)])
def test_aggregate_vs_oracle(B, C, H, W):
    from centernet_b200 import decode as D
    heat = noise(B, C, H, W, 9, bias=0.5)
    d, = dev(heat)
    np.testing.assert_array_equal(D._h_aggregate(d, 0.1).cpu().numpy(), O.h_aggregate(heat, 0.1))
    np.testing.assert_array_equal(D._v_aggregate(d, 0.1).cpu().numpy(), O.v_aggregate(heat, 0.1))
    np.testing.assert_array_equal(D._left_aggregate(d).cpu().numpy(), O.left_aggregate(heat))
    np.testing.assert_array_equal(D._bottom_aggregate(d).cpu().numpy(), O.bottom_aggregate(heat))
    np.testing.assert_array_equal(D._right_aggregate(d).cpu().numpy(), O.right_aggregate(heat))
    np.testing.assert_array_equal(D._top_aggregate(d).cpu().numpy(), O.top_aggregate(heat))
    np.testing.assert_array_equal(d.cpu().numpy(), heat)


# ------------------------------------------------------------------ focal loss / splat / reg losses
def test_golden_losses():
    from centernet_b200 import losses as L
    g = golden("losses")
    pred, gt, logits = dev(g["pred"], g["gt"], g["logits"])
    p = pred.clone().requires_grad_(True)
    loss = L.FocalLoss()(p, gt)
    loss.backward()
    np.testing.assert_allclose(loss.item(), g["neg_loss"], rtol=1e-5)                 # SURVEY 8d: rel 1e-5
    np.testing.assert_allclose(p.grad.cpu().numpy(), g["neg_loss_grad"], rtol=1e-4, atol=1e-5)
    loss0 = L._neg_loss(pred, torch.clamp(gt, max=0.5))
    np.testing.assert_allclose(loss0.item(), g["neg_loss_nopos"], rtol=1e-5)
    # fused _sigmoid + loss from the raw logits, gradient w.r.t. the logits via autograd of the reference formula
    lg = logits.clone().requires_grad_(True)
    lf = L._neg_loss_from_logits(lg, gt)
    lf.backward()
    np.testing.assert_allclose(lf.item(), g["neg_loss"], rtol=2e-5)
    ref_l = logits.clone().requires_grad_(True)
    pr = torch.clamp(torch.sigmoid(ref_l), 1e-4, 1 - 1e-4)
    pos = (gt == 1).float(); neg = (gt < 1).float()
    ref = -((torch.log(pr) * (1 - pr) ** 2 * pos).sum() + (torch.log(1 - pr) * pr ** 2 * (1 - gt) ** 4 * neg).sum()) / pos.sum()
    ref.backward()
    np.testing.assert_allclose(lg.grad.cpu().numpy(), ref_l.grad.cpu().numpy(), rtol=1e-3, atol=1e-6)
    # regression losses
    output, ind, target, wmask = dev(g["output"], g["ind"], g["target"], g["wmask"])
    mask = torch.from_numpy(g["mask"]).cuda()
    for cls, key, tgt, m in ((L.RegL1Loss, "reg_l1", target, mask), (L.RegLoss, "reg_sl1", target, mask),
                             (L.NormRegL1Loss, "norm_l1", target.abs() + 0.5, mask),
                             (L.RegWeightedL1Loss, "weighted_l1", target, wmask)):
        o = output.clone().requires_grad_(True)
        val = cls()(o, m, ind, tgt)
        np.testing.assert_allclose(val.item(), g[key], rtol=1e-5, err_msg=key)
        val.backward()
        assert torch.isfinite(o.grad).all()
    # RegL1Loss gradient against autograd of the reference formula
    o = output.clone().requires_grad_(True)
    L.RegL1Loss()(o, mask, ind, target).backward()
    o2 = output.clone().requires_grad_(True)
    B, D_ = o2.shape[:2]
    predt = o2.view(B, D_, -1).permute(0, 2, 1).gather(1, ind.unsqueeze(2).expand(B, ind.size(1), D_))
    mm = mask.unsqueeze(2).expand_as(predt).float()
    (torch.nn.functional.l1_loss(predt * mm, target * mm, reduction="sum") / (mm.sum() + 1e-4)).backward()
    np.testing.assert_allclose(o.grad.cpu().numpy(), o2.grad.cpu().numpy(), rtol=1e-5, atol=1e-7)


def test_golden_splat_and_fused_focal():
    from centernet_b200 import losses as L
    g = golden("splat")
    C, H, W = int(g["C"]), int(g["H"]), int(g["W"])
    cls, cx, cy, rad, val = dev(g["obj_cls"], g["obj_cx"], g["obj_cy"], g["obj_radius"], g["obj_valid"])
    hm = L.splat_gaussian(cls, cx, cy, rad, val, C, H, W)
    np.testing.assert_array_equal(hm.cpu().numpy(), g["hm"])
    assert np.array_equal(hm.cpu().numpy() == 1.0, g["hm"] == 1.0)           # identical positive set
    # fused splat+focal == focal on the dense reference target
    B = cls.shape[0]
    pred = torch.from_numpy(losses_np.sigmoid_clamped(rnd((B, C, H, W), 3, 2.0, normal=True) - 2)).cuda()
    want, npos = losses_np.neg_loss(pred.cpu().numpy(), g["hm"])
    p = pred.clone().requires_grad_(True)
    loss = L.FocalSplatLoss()(p, cls, cx, cy, rad, val)
    loss.backward()
    np.testing.assert_allclose(loss.item(), want, rtol=1e-5)
    np.testing.assert_allclose(p.grad.cpu().numpy(), losses_np.neg_loss_grad(pred.cpu().numpy(), g["hm"]),
                               rtol=1e-4, atol=1e-6)


def test_focal_full_size_linearity():
    """BASELINE configs[1] size: loss(pred, gt) from two half batches recombines (linearity of the sums)."""
    from centernet_b200 import losses as L
    B, C, H, W, M = 8, 80, 128, 128, 32
    g = torch.Generator(device="cuda").manual_seed(5)
    pred = torch.clamp(torch.sigmoid(torch.randn(B, C, H, W, device="cuda", generator=g) - 2.19), 1e-4, 1 - 1e-4)
    cls = torch.randint(0, C, (B, M), device="cuda", generator=g)
    cx = torch.randint(0, W, (B, M), device="cuda", generator=g); cy = torch.randint(0, H, (B, M), device="cuda", generator=g)
    rad = torch.randint(0, 12, (B, M), device="cuda", generator=g)
    val = torch.ones(B, M, dtype=torch.uint8, device="cuda")
    gt = L.splat_gaussian(cls, cx, cy, rad, val, C, H, W)
    want = image_np.splat_objects(*[t.cpu().numpy() for t in (cls, cx, cy, rad, val)], C, H, W)
    np.testing.assert_array_equal(gt.cpu().numpy(), want)
    full = L._neg_loss(pred, gt)
    fused = L.FocalSplatLoss()(pred, cls, cx, cy, rad, val)
    np.testing.assert_allclose(full.item(), fused.item(), rtol=1e-6)
    n = float((gt == 1).sum())
    n1 = float((gt[:4] == 1).sum()); n2 = n - n1
    a = L._neg_loss(pred[:4].contiguous(), gt[:4].contiguous()).item() * n1
    b = L._neg_loss(pred[4:].contiguous(), gt[4:].contiguous()).item() * n2
    np.testing.assert_allclose((a + b) / n, full.item(), rtol=1e-5)
    ref, _ = losses_np.neg_loss(pred.cpu().numpy(), gt.cpu().numpy())
    np.testing.assert_allclose(full.item(), ref, rtol=1e-5)
