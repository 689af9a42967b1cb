"""N2: detection post-processing (utils/post_process.py:83-114, external/nms.pyx:77-275, detectors/ctdet.py:76-92).
tests/golden/post.npz holds outputs of the UNMODIFIED reference (post_process.py imported, nms.pyx compiled by
oracle/build_ref.py).  CPU half pins the numpy oracle; GPU half checks the CUDA path bit for bit."""
import numpy as np
import pytest
import torch

from helpers import golden
from oracle import post_np as O

NMS_CASES = ("g", "lin", "hard", "g1", "gbig")


def flat(res, B, C):
    rows = []
    for i in range(B):
        for j in range(1, C + 1):
            a = np.asarray(res[i][j], np.float32).reshape(-1, 5)
            rows.append(np.concatenate([np.full((len(a), 1), i, np.float32), np.full((len(a), 1), j, np.float32), a], 1))
    return np.concatenate(rows, 0)


# --------------------------------------------------------------------------- CPU: oracle vs reference golden
def test_oracle_post_process():
    g = golden("post")
    np.testing.assert_array_equal(flat(O.ctdet_post_process(g["ct_dets"], g["ct_c"], g["ct_s"], 128, 128, 80), 2, 80),
                                  g["ct_rows"])
    np.testing.assert_array_equal(flat(O.ctdet_post_process(g["ct_dets"], g["ct_c"], g["ct_s2"], 120, 160, 80), 2, 80),
                                  g["ct_rows2"])
    r = O.multi_pose_post_process(g["mp_dets"], g["ct_c"], g["ct_s"], 128, 128)
    np.testing.assert_array_equal(np.stack([r[i][1] for i in range(2)]), g["mp_rows"])


@pytest.mark.parametrize("name", NMS_CASES)
def test_oracle_soft_nms(name):
    g = golden("post")
    a = g["nms_%s_in" % name].copy(); cfg = g["nms_%s_cfg" % name]
    n = O.soft_nms(a, sigma=cfg[0], Nt=cfg[1], threshold=cfg[2], method=int(cfg[3]))
    assert n == int(g["nms_%s_n" % name])
    np.testing.assert_array_equal(a, g["nms_%s_out" % name])      # the whole array, stale rows included


def test_oracle_soft_nms_39_and_merge():
    g = golden("post")
    a = g["nms39_in"].copy()
    assert O.soft_nms(a, Nt=0.5, method=2, ncols_swap=34) == int(g["nms39_n"])
    np.testing.assert_array_equal(a, g["nms39_out"])
    scales = [{j: g["mg_s%d_c%d" % (si, j)] for j in range(1, 6)} for si in range(2)]
    res = O.merge_outputs(scales, 5, 100)
    for j in range(1, 6):
        np.testing.assert_array_equal(res[j], g["mg_out_c%d" % j])


def test_reference_nms_module_if_built():
    """The oracle against the compiled reference soft_nms on three random 70-box lists (gaussian, linear, hard):
    tests/golden/nms_lists.npz holds what the reference module returned for them (make_golden_nms.py)."""
    g = golden("nms_lists")
    for i in range(3):
        method, Nt = g["cfg%d" % i]
        a = g["in%d" % i].copy()
        assert O.soft_nms(a, Nt=float(Nt), method=int(method)) == int(g["n%d" % i])
        np.testing.assert_array_equal(a, g["out%d" % i])


# --------------------------------------------------------------------------- GPU: the CUDA path
@pytest.mark.gpu
def test_gpu_post_process():
    from centernet_b200 import post_process as P
    g = golden("post")
    for dets in (g["ct_dets"], torch.from_numpy(g["ct_dets"]).cuda()):      # numpy (reference form) and CUDA tensor
        r = P.ctdet_post_process(dets, g["ct_c"], g["ct_s"], 128, 128, 80)
        assert isinstance(r[0][1], list)
        np.testing.assert_array_equal(flat(r, 2, 80), g["ct_rows"])
    r = P.ctdet_post_process(g["ct_dets"], g["ct_c"], g["ct_s2"], 120, 160, 80)
    np.testing.assert_array_equal(flat(r, 2, 80), g["ct_rows2"])
    r = P.multi_pose_post_process(torch.from_numpy(g["mp_dets"]).cuda(), g["ct_c"], g["ct_s"], 128, 128)
    np.testing.assert_array_equal(np.stack([np.asarray(r[i][1], np.float32) for i in range(2)]), g["mp_rows"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", NMS_CASES)
def test_gpu_soft_nms(name):
    from centernet_b200 import post_process as P
    g = golden("post")
    a = g["nms_%s_in" % name].copy(); cfg = g["nms_%s_cfg" % name]
    keep = P.soft_nms(a, sigma=float(cfg[0]), Nt=float(cfg[1]), threshold=float(cfg[2]), method=int(cfg[3]))
    assert keep == list(range(int(g["nms_%s_n" % name])))
    np.testing.assert_array_equal(a, g["nms_%s_out" % name])


@pytest.mark.gpu
def test_gpu_soft_nms_39_and_merge():
    from centernet_b200 import post_process as P
    g = golden("post")
    a = g["nms39_in"].copy()
    assert len(P.soft_nms_39(a, Nt=0.5, method=2)) == int(g["nms39_n"])
    np.testing.assert_array_equal(a, g["nms39_out"])
    # merge_outputs on the device: rebuild [1, n, 6] decode-like tensors for the two scales (identity back-projection:
    # centre = (w/2, h/2), scale = w), class column from the golden's per-class lists
    dets = []
    for si in range(2):
        rows = [np.concatenate([g["mg_s%d_c%d" % (si, j)], np.full((len(g["mg_s%d_c%d" % (si, j)]), 1), j - 1, np.float32)], 1)
                for j in range(1, 6)]
        dets.append(torch.from_numpy(np.concatenate(rows, 0)[None]).cuda())
    meta = {"c": [np.array([64.0, 64.0], np.float32)], "s": [128.0], "out_height": 128, "out_width": 128}
    res = P.ctdet_merge_device(dets, [meta, meta], 5, max_per_image=100)
    for j in range(1, 6):
        np.testing.assert_array_equal(res[0][j], g["mg_out_c%d" % j])


@pytest.mark.gpu
def test_gpu_merge_vs_oracle_multi_image():
    """Two images x two scales straight from ctdet_decode-shaped tensors, against the oracle pipeline."""
    from centernet_b200 import post_process as P
    rng = np.random.default_rng(12)
    B, K, C = 2, 100, 80
    metas, dets = [], []
    for sc in (1.0, 1.5):
        d = np.zeros((B, K, 6), np.float32)
        d[..., 0] = rng.uniform(0, 100, (B, K)); d[..., 1] = rng.uniform(0, 100, (B, K))
        d[..., 2] = d[..., 0] + rng.uniform(2, 40, (B, K)); d[..., 3] = d[..., 1] + rng.uniform(2, 40, (B, K))
        d[..., 4] = np.sort(rng.uniform(0, 1, (B, K)), axis=1)[:, ::-1]
        d[..., 5] = rng.integers(0, 6, (B, K))        # few classes -> long per-class lists
        dets.append(d)
        metas.append({"c": [np.array([300.0 * sc, 200.0 * sc], np.float32)] * B, "s": [640.0 * sc] * B,
                      "out_height": 128, "out_width": 128, "scale": sc})
    got = P.ctdet_merge_device([torch.from_numpy(d).cuda() for d in dets], metas, C, max_per_image=100)
    for i in range(B):
        per_scale = []
        for d, m in zip(dets, metas):
            r = O.ctdet_post_process(d[i:i + 1], m["c"][:1], m["s"][:1], 128, 128, C)[0]
            for j in r:
                r[j] = np.asarray(r[j], np.float32).reshape(-1, 5)
                r[j][:, :4] /= m["scale"]
            per_scale.append(r)
        want = O.merge_outputs(per_scale, C, 100)
        for j in range(1, C + 1):
            np.testing.assert_array_equal(got[i][j], want[j])
