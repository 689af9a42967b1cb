"""GPU: everything DCNv2 / deformable-PSROI pinned to THE REFERENCE ITSELF -- the reference's own two .cu
files compiled unmodified for sm_100a (oracle/build_ref.py) under a cuBLAS restatement of the THC host loop
(oracle/ref_host.cu), run on a B200 on the seeded inputs below.  tests/golden/ref_gpu.npz keeps what it
returned (tests/golden/make_golden_ref_gpu.py): whole tensors up to SAMPLE elements, SAMPLE fixed positions
spread over larger ones (sample_positions) and their abs max.  Three-way: the fp64 restatement
(oracle/dcn_ref.py), the numpy restatement (oracle/psroi_np.py) and our kernels are each held to it.
Tolerances: forward <= 1e-4 abs (north_star), backward at DCNv2/test.py:90,115 (atol 1e-3, scaled)."""
import numpy as np
import pytest
import torch

from helpers import golden
from oracle import dcn_ref, psroi_np

pytestmark = pytest.mark.gpu

SAMPLE = 512           # elements kept per reference output
PROBE = 16             # leading elements kept per input: catches a drift of the seeded generators
STRIDE = 2654435761    # prime, so i * STRIDE mod n visits SAMPLE distinct positions scattered over the tensor


def sample_positions(n):
    return np.arange(n) if n <= SAMPLE else np.sort(np.arange(SAMPLE, dtype=np.int64) * STRIDE % n)


def make(B, Ci, H, W, Co, dg, stride=1, seed=0, off_scale=2.0):
    g = torch.Generator().manual_seed(seed)
    Ho = (H + 2 - 3) // stride + 1
    Wo = (W + 2 - 3) // stride + 1
    x = torch.randn(B, Ci, H, W, generator=g)
    off = torch.randn(B, 18 * dg, Ho, Wo, generator=g) * off_scale
    m = torch.sigmoid(torch.randn(B, 9 * dg, Ho, Wo, generator=g))
    w = torch.randn(Co, Ci, 3, 3, generator=g) / (3.0 * Ci ** 0.5)
    b = torch.randn(Co, generator=g)
    return x, off, m, w, b


def kat_inputs():
    """DCNv2/test.py:32-65: identity weights, zero offsets, mask 0.5 -> 2 * out == x."""
    N, C, H, W = 2, 2, 4, 4
    x = torch.randn(N, C, H, W, generator=torch.Generator().manual_seed(1))
    w = torch.zeros(C, C, 3, 3)
    for i in range(C):
        w[i, i, 1, 1] = 1.0
    return x, torch.zeros(N, 18, H, W), torch.full((N, 9, H, W), 0.5), w, torch.zeros(C)


# BASELINE configs[1] (dla_34 512x512) DCN layer shapes (SURVEY 3.2) + odd / strided / grouped cases
LAYERS = [
    # B, Cin, H, W, Cout, dg, stride
    (2, 64, 128, 128, 64, 1, 1),
    (2, 128, 64, 64, 128, 1, 1),
    (2, 256, 32, 32, 256, 1, 1),
    (2, 512, 16, 16, 256, 1, 1),
    (2, 128, 64, 64, 64, 1, 1),
    (2, 256, 32, 32, 128, 1, 1),
    (2, 64, 32, 32, 64, 2, 1),
    (2, 12, 9, 11, 5, 2, 1),
    (2, 6, 10, 14, 7, 1, 2),
]
FP32_LAYERS = [(2, 64, 128, 128, 64, 1, 1), (2, 512, 16, 16, 256, 1, 1)]
BWD_LAYERS = [(2, 64, 64, 64, 64, 1, 1), (2, 128, 32, 32, 128, 1, 1), (2, 256, 16, 16, 256, 1, 1),
              (1, 512, 16, 16, 256, 1, 1), (2, 64, 16, 16, 64, 2, 1), (1, 12, 9, 11, 5, 2, 1), (2, 6, 10, 14, 7, 1, 2)]
GRADS = ("input", "offset", "mask", "weight", "bias")


def bwd_inputs(B, Ci, H, W, Co, dg, stride):
    x, off, m, w, b = make(B, Ci, H, W, Co, dg, stride, seed=3, off_scale=1.3)
    Ho = (H + 2 - 3) // stride + 1; Wo = (W + 2 - 3) // stride + 1
    go = torch.randn(B, Co, Ho, Wo, generator=torch.Generator().manual_seed(9))
    return (x, off, m, w, b), go


def key(kind, cfg):
    return kind + "_" + "_".join(str(v) for v in cfg)


# ---------------------------------------------------------------- golden access
_G = None


def ref():
    global _G
    if _G is None:
        _G = golden("ref_gpu")
    return _G


def check_inputs(k, *tensors):
    g = ref()
    for i, t in enumerate(tensors):
        if t is None:
            continue
        lead = t.detach().reshape(-1)[:PROBE].cpu().numpy()
        np.testing.assert_allclose(lead, g["%s__in%d" % (k, i)], rtol=0, atol=1e-6,
                                   err_msg="%s: seeded inputs differ from those the golden was made from" % k)


def sampled(t, k):
    """t at the positions the golden kept for output k, as float64 numpy."""
    g = ref()
    assert tuple(t.shape) == tuple(g[k + "__shape"]), (k, tuple(t.shape), tuple(g[k + "__shape"]))
    flat = t.detach().reshape(-1)
    idx = torch.from_numpy(sample_positions(flat.numel())).to(flat.device)
    return flat[idx].double().cpu().numpy()


def want(k):
    return ref()[k + "__val"].astype(np.float64)


def absmax(k):
    return float(ref()[k + "__absmax"])


def err(t, k):
    return float(np.abs(sampled(t, k) - want(k)).max())


def check_whole(got, orc, k, atol, rtol=0.0, what=""):
    """The golden keeps a sample of the reference: every element of the kernel's output is held to the oracle
    instead, and the kernel's abs max to the reference's."""
    a = got.detach().double().cpu(); o = torch.as_tensor(orc).detach().double().cpu()
    assert a.shape == o.shape, (what, a.shape, o.shape)
    bad = ((a - o).abs() > atol + rtol * o.abs()).sum().item()
    assert bad == 0, (what, k, "kernel vs oracle: %d elements off, max err %g" % (bad, (a - o).abs().max().item()))
    d = abs(a.abs().max().item() - absmax(k))
    assert d <= atol + rtol * absmax(k), (what, k, "abs max vs reference", d)


# ---------------------------------------------------------------- DCNv2
def test_reference_zero_offset_kat_on_ref():
    """DCNv2/test.py:32-65 on the compiled reference (sanity of the host-loop restatement), and our kernel on the
    same inputs."""
    from centernet_b200.dcn_v2_func import DCNv2Function
    x, off, m, w, b = kat_inputs()
    check_inputs("kat", x)
    assert np.abs(want("kat") * 2 - x.double().numpy().reshape(-1)).max() < 1e-7
    got = DCNv2Function(1, 1, 1, 1)(*[t.cuda() for t in (x, off, m, w, b)])
    assert err(got, "kat") <= 1e-6


@pytest.mark.parametrize("B,Ci,H,W,Co,dg,stride", LAYERS)
def test_forward_three_way(B, Ci, H, W, Co, dg, stride):
    from centernet_b200.dcn_v2_func import DCNv2Function
    k = key("fwd", (B, Ci, H, W, Co, dg, stride))
    x, off, m, w, b = make(B, Ci, H, W, Co, dg, stride)
    check_inputs(k, x, off, m, w, b)
    cu = [t.cuda() for t in (x, off, m, w, b)]
    got = DCNv2Function(stride, 1, 1, dg)(*cu)          # tcgen05 (3xTF32) path
    torch.cuda.synchronize()
    e = err(got, k)
    assert e <= 1e-4, ("kernel vs reference", e)
    orc = dcn_ref.dcn_v2_forward(x, off, m, w, b, stride, 1, 1, dg)
    e_o = err(orc, k)
    assert e_o <= 1e-4, ("fp64 oracle vs reference", e_o)
    check_whole(got, orc, k, 1e-4)


@pytest.mark.parametrize("B,Ci,H,W,Co,dg,stride", FP32_LAYERS)
def test_forward_fp32_path_vs_reference(B, Ci, H, W, Co, dg, stride):
    """cnb_dcnv2_forward without a workspace = the fp32 CUDA-core contraction."""
    from centernet_b200._lib import C, ptr, stream_ptr
    k = key("fp32", (B, Ci, H, W, Co, dg, stride))
    inputs = make(B, Ci, H, W, Co, dg, stride, seed=5)
    check_inputs(k, *inputs)
    x, off, m, w, b = [t.cuda() for t in inputs]
    Ho = (H + 2 - 3) // stride + 1; Wo = (W + 2 - 3) // stride + 1
    out = torch.empty(B, Co, Ho, Wo, device="cuda")
    C.dcnv2_forward(ptr(x), ptr(off), ptr(m), ptr(w), ptr(b), ptr(out), B, Ci, H, W, Co, 3, 3, stride, stride, 1, 1, 1, 1,
                    dg, 0, 0, stream_ptr(x))
    assert err(out, k) <= 1e-4
    check_whole(out, dcn_ref.dcn_v2_forward(*inputs, stride, 1, 1, dg), k, 1e-4)


@pytest.mark.parametrize("B,Ci,H,W,Co,dg,stride", BWD_LAYERS)
def test_backward_three_way(B, Ci, H, W, Co, dg, stride):
    from centernet_b200.dcn_v2_func import DCNv2Function
    k = key("bwd", (B, Ci, H, W, Co, dg, stride))
    (x, off, m, w, b), go = bwd_inputs(B, Ci, H, W, Co, dg, stride)
    check_inputs(k, x, off, m, w, b, go)
    cu = [t.cuda() for t in (x, off, m, w, b)]
    cl = [t.clone().requires_grad_(True) for t in cu]
    (DCNv2Function(stride, 1, 1, dg)(*cl) * go.cuda()).sum().backward()
    leaves = [t.clone().double().requires_grad_(True) for t in (x, off, m, w, b)]
    (dcn_ref.dcn_v2_forward(*leaves, stride, 1, 1, dg) * go.double()).sum().backward()
    for name, a, o in zip(GRADS, cl, leaves):
        kk = k + "_" + name
        scale = max(1.0, absmax(kk))
        e = err(a.grad, kk)
        assert e <= 1e-3 * scale, ("kernel vs reference", name, e, scale)
        e_o = err(o.grad, kk)
        assert e_o <= 1e-3 * scale, ("fp64 oracle vs reference", name, e_o, scale)
        check_whole(a.grad, o.grad, kk, 1e-3 * scale, what=name)


# ---------------------------------------------------------------- deformable PSROI pooling (N4)
def _case(seed, B, C, H, W, N, output_dim, group, pooled, part, spp, classes, trans_std, no_trans):
    rng = np.random.default_rng(seed)
    data = rng.standard_normal((B, C, H, W)).astype(np.float32)
    x = rng.uniform(-6, W * 4 - 8, N); y = rng.uniform(-6, H * 4 - 8, N)
    w = rng.uniform(1, W * 3, N); h = rng.uniform(1, H * 3, N)
    rois = np.stack([rng.integers(0, B, N).astype(np.float64), x, y, x + w, y + h], 1).astype(np.float32)
    trans = None if no_trans else rng.standard_normal((N, 2 * classes, part, part)).astype(np.float32)
    cfg = dict(no_trans=no_trans, spatial_scale=0.25, output_dim=output_dim, group_size=group, pooled_size=pooled,
               part_size=part, sample_per_part=spp, trans_std=trans_std)
    return data, rois, trans, cfg


def psroi_kwargs(cfg):
    return dict(spatial_scale=cfg["spatial_scale"], pooled_size=cfg["pooled_size"], output_dim=cfg["output_dim"],
                no_trans=cfg["no_trans"], group_size=cfg["group_size"], part_size=cfg["part_size"],
                sample_per_part=cfg["sample_per_part"], trans_std=cfg["trans_std"])


def psroi_grad_out(shape):
    return np.random.default_rng(9).standard_normal(tuple(shape)).astype(np.float32)


PS_CASES = [
    (1, 2, 8, 9, 9, 5, 2, 2, 3, 3, 2, 2, 0.1, False),
    (2, 2, 18, 12, 10, 6, 2, 3, 4, 2, 3, 1, 0.3, False),
    (3, 1, 4, 7, 7, 4, 4, 1, 3, 3, 4, 2, 0.0, False),
    (4, 3, 16, 16, 16, 7, 16, 1, 7, 7, 4, 1, 0.1, True),
    (5, 2, 98, 20, 24, 12, 2, 7, 7, 7, 4, 1, 0.1, False),    # DCNv2/test.py:148-166 style: group 7, 7x7 bins
]


@pytest.mark.parametrize("case", PS_CASES)
def test_psroi_three_way(case):
    from centernet_b200.dcn_v2_func import DCNv2PoolingFunction
    k = "psroi_%d" % case[0]
    data, rois, trans, cfg = _case(*case)
    check_inputs(k, torch.from_numpy(data), torch.from_numpy(rois), None if trans is None else torch.from_numpy(trans))
    d = torch.from_numpy(data).cuda(); r = torch.from_numpy(rois).cuda()
    t = torch.zeros(1, device="cuda") if trans is None else torch.from_numpy(trans).cuda()
    go_np = psroi_grad_out(ref()[k + "_out__shape"])
    go = torch.from_numpy(go_np).cuda()
    # numpy restatement vs the reference
    out_np, cnt = psroi_np.psroi_forward(data, rois, trans, **cfg)
    np.testing.assert_allclose(sampled(torch.from_numpy(out_np), k + "_out"), want(k + "_out"), rtol=0, atol=1e-5)
    np.testing.assert_array_equal(sampled(torch.from_numpy(cnt), k + "_cnt"), want(k + "_cnt"))
    gd, gt = psroi_np.psroi_backward(go_np, data, rois, trans, cnt, **cfg)
    np.testing.assert_allclose(sampled(torch.from_numpy(gd), k + "_gi"), want(k + "_gi"), rtol=1e-4, atol=1e-4)
    if trans is not None:
        np.testing.assert_allclose(sampled(torch.from_numpy(gt), k + "_gt"), want(k + "_gt"), rtol=1e-4, atol=1e-4)
    # our kernels vs the reference
    fn = DCNv2PoolingFunction(cfg["spatial_scale"], cfg["pooled_size"], cfg["output_dim"], cfg["no_trans"],
                              cfg["group_size"], cfg["part_size"], cfg["sample_per_part"], cfg["trans_std"])
    dd = d.clone().requires_grad_(True)
    tt = d.new() if trans is None else t.clone().requires_grad_(True)
    out = fn(dd, r, tt)
    # same expression order; nvcc contracts a few multiply-adds differently in the two builds: a handful of ulps
    assert err(out, k + "_out") <= 2e-5
    out.backward(go)
    np.testing.assert_allclose(sampled(dd.grad, k + "_gi"), want(k + "_gi"), rtol=1e-4, atol=1e-4)
    if trans is not None:
        np.testing.assert_allclose(sampled(tt.grad, k + "_gt"), want(k + "_gt"), rtol=1e-4, atol=1e-4)
    # whole tensors against the numpy restatement: the sums of the two bounds each is held to above
    check_whole(out, out_np, k + "_out", 3e-5, what="out")
    check_whole(dd.grad, gd, k + "_gi", 2e-4, 2e-4, what="grad input")
    if trans is not None:
        check_whole(tt.grad, gt, k + "_gt", 2e-4, 2e-4, what="grad trans")
