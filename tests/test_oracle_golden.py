"""CPU: the numpy oracle reproduces the outputs of the unmodified reference
(tests/golden/*.npz, made by tests/golden/make_golden.py) -- this is what pins it."""
import numpy as np

from helpers import assert_dets_equal, golden
from oracle import decode_np as O
from oracle import image_np, losses_np


def test_raw_ops():
    g = golden("raw_ops")
    K = int(g["K"])
    nms = O.nms(g["heat"])
    np.testing.assert_array_equal(nms, g["nms"])
    s, inds, clses, ys, xs = O.topk(nms, K)
    for got, key in ((s, "topk_scores"), (inds, "topk_inds"), (clses, "topk_clses"), (ys, "topk_ys"), (xs, "topk_xs")):
        np.testing.assert_array_equal(got, g[key])
    cs, ci, cy, cx = O.topk_channel(nms, K)
    for got, key in ((cs, "ch_scores"), (ci, "ch_inds"), (cy, "ch_ys"), (cx, "ch_xs")):
        np.testing.assert_array_equal(got, g[key])


def test_ctdet():
    g = golden("ctdet_noise")
    K = int(g["K"])
    np.testing.assert_array_equal(O.ctdet_decode(g["heat"], g["wh"], g["reg"], K=K), g["dets"])
    np.testing.assert_array_equal(O.ctdet_decode(g["heat"], g["wh"], None, K=K), g["dets_noreg"])
    g = golden("ctdet_blobs_catspec")
    np.testing.assert_array_equal(O.ctdet_decode(g["heat"], g["wh"], g["reg"], cat_spec_wh=True, K=int(g["K"])),
                                  g["dets"])


def test_ctdet_ties_and_fillers():
    g = golden("ctdet_ties")
    got = O.ctdet_decode(g["heat"], g["wh"], g["reg"], K=int(g["K"]))
    assert_dets_equal(g["dets"], got, positive_only=True, what="ctdet_ties")
    # the oracle's own tie rule: equal scores come out in flat-index order
    assert got[0, 0, 4] == np.float32(0.7)
    assert list(got[0, 1:4, 5]) == [0.0, 0.0, 1.0]


def test_multi_pose():
    g = golden("multi_pose")
    K = int(g["K"])
    a = (g["heat"], g["wh"], g["kps"])
    np.testing.assert_array_equal(O.multi_pose_decode(*a, g["reg"], g["hm_hp"], g["hp_offset"], K=K), g["dets"])
    np.testing.assert_array_equal(O.multi_pose_decode(*a, None, g["hm_hp"], None, K=K), g["dets_nooff"])
    np.testing.assert_array_equal(O.multi_pose_decode(*a, g["reg"], K=K), g["dets_nohp"])


def test_ddd():
    g = golden("ddd")
    K = int(g["K"])
    np.testing.assert_array_equal(
        O.ddd_decode(g["heat"], g["rot"], g["depth"], g["dim"], g["wh"], g["reg"], K=K), g["dets"])
    np.testing.assert_array_equal(O.ddd_decode(g["heat"], g["rot"], g["depth"], g["dim"], K=K), g["dets_min"])


def test_aggregate():
    g = golden("aggregate")
    for name, fn in (("left", O.left_aggregate), ("right", O.right_aggregate), ("top", O.top_aggregate),
                     ("bottom", O.bottom_aggregate)):
        np.testing.assert_array_equal(fn(g["heat"]), g[name])
    np.testing.assert_array_equal(O.h_aggregate(g["heat"], 0.1), g["h"])
    np.testing.assert_array_equal(O.v_aggregate(g["heat"], 0.1), g["v"])


def test_exct():
    g = golden("exct")
    K, ND = int(g["K"]), int(g["num_dets"])
    maps = (g["t"], g["l"], g["b"], g["r"], g["ct"])
    regs = (g["t_regr"], g["l_regr"], g["b_regr"], g["r_regr"])
    assert_dets_equal(g["dets"], O.exct_decode(*maps, *regs, K=K, num_dets=ND), positive_only=True, what="exct")
    assert_dets_equal(g["dets_noreg"], O.exct_decode(*maps, K=K, num_dets=ND), positive_only=True, what="exct_noreg")
    assert_dets_equal(g["dets_aggr"], O.exct_decode(*maps, *regs, K=K, num_dets=ND, aggr_weight=0.1),
                      positive_only=True, what="exct_aggr")
    agn = O.agnex_ct_decode(g["t1"], g["l1"], g["b1"], g["r1"], g["ct"], *regs, K=K, num_dets=ND)
    assert_dets_equal(g["dets_agn"], agn, positive_only=True, what="agnex")


def test_losses():
    g = golden("losses")
    np.testing.assert_allclose(losses_np.sigmoid_clamped(g["logits"]), g["pred"], rtol=1e-6, atol=1e-7)
    loss, npos = losses_np.neg_loss(g["pred"], g["gt"])
    assert npos == float(g["num_pos"]) and npos > 0
    np.testing.assert_allclose(loss, g["neg_loss"], rtol=1e-5)
    np.testing.assert_allclose(losses_np.neg_loss_grad(g["pred"], g["gt"]), g["neg_loss_grad"], rtol=1e-4, atol=1e-6)
    loss0, npos0 = losses_np.neg_loss(g["pred"], np.minimum(g["gt"], 0.5))
    assert npos0 == 0
    np.testing.assert_allclose(loss0, g["neg_loss_nopos"], rtol=1e-5)
    # gradient w.r.t. the logit: float64 autograd of _sigmoid (clamp(sigmoid(x))) + _neg_loss.  The logits x4 put
    # part of the map outside the clamp, where the gradient must be exactly 0.
    import torch
    gt = torch.from_numpy(g["gt"]).double()
    for scale in (1.0, 4.0):
        x32 = g["logits"] * np.float32(scale)
        x = torch.from_numpy(x32).double().requires_grad_(True)
        pr = torch.clamp(torch.sigmoid(x), 1e-4, 1 - 1e-4)
        pos, neg = (gt == 1).double(), (gt < 1).double()
        ref = -((torch.log(pr) * (1 - pr) ** 2 * pos).sum()
                + (torch.log(1 - pr) * pr ** 2 * (1 - gt) ** 4 * neg).sum()) / pos.sum()
        ref.backward()
        want = x.grad.numpy()
        s32 = (1 / (1 + np.exp(-x32.astype(np.float64)))).astype(np.float32)
        got = losses_np.neg_loss_grad_logits(s32, g["gt"])
        assert got.dtype == np.float64
        np.testing.assert_array_equal(got == 0, want == 0)
        assert (want == 0).any() == (scale > 1)
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-6 * np.abs(want).max())
    a = (g["output"], g["mask"], g["ind"], g["target"])
    np.testing.assert_allclose(losses_np.reg_l1_loss(*a), g["reg_l1"], rtol=1e-5)
    np.testing.assert_allclose(losses_np.reg_loss(*a), g["reg_sl1"], rtol=1e-5)
    np.testing.assert_allclose(
        losses_np.norm_reg_l1_loss(g["output"], g["mask"], g["ind"], np.abs(g["target"]) + 0.5), g["norm_l1"],
        rtol=1e-5)
    np.testing.assert_allclose(losses_np.reg_weighted_l1_loss(g["output"], g["wmask"], g["ind"], g["target"]),
                               g["weighted_l1"], rtol=1e-5)


def test_splat():
    g = golden("splat")
    hm = image_np.splat_objects(g["obj_cls"], g["obj_cx"], g["obj_cy"], g["obj_radius"], g["obj_valid"],
                                int(g["C"]), int(g["H"]), int(g["W"]))
    np.testing.assert_array_equal(hm, g["hm"])
    for b in range(g["box_h"].shape[0]):
        for m in range(g["box_h"].shape[1]):
            r = max(0, int(image_np.gaussian_radius((np.ceil(g["box_h"][b, m]), np.ceil(g["box_w"][b, m])))))
            assert r == g["obj_radius"][b, m]
    # SURVEY appendix A facts
    assert int(image_np.gaussian_radius((10, 20))) == 3 and int(image_np.gaussian_radius((1, 1))) == 0
    assert image_np.gaussian2d(7, 7 / 6)[3, 3] == 1.0


def test_timed_cpu_port_reproduces_the_reference():
    """oracle/torch_port.py is what bench.py times as the reference's CPU path; it must give the reference's numbers
    (tools/compare_port_with_reference.py checks it against the live reference in the build container)."""
    import torch
    from oracle import torch_port
    g = golden("ctdet_noise")
    K = int(g["K"])
    heat, wh, reg = (torch.from_numpy(g[k]) for k in ("heat", "wh", "reg"))
    np.testing.assert_array_equal(torch_port.ctdet_decode(heat.clone(), wh, reg=reg, K=K).numpy(), g["dets"])
    np.testing.assert_array_equal(torch_port.ctdet_decode(heat.clone(), wh, reg=None, K=K).numpy(), g["dets_noreg"])
