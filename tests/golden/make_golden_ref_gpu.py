"""Generates tests/golden/ref_gpu.npz: the reference's own DCNv2 / deformable-PSROI CUDA kernels (oracle/_ref,
built by oracle/build_ref.py from the reference sources) on the seeded inputs of tests/test_ref_gpu.py.  Needs a
B200 and the prebuilt oracle/_ref/libdcnv2_ref.so:
    python tests/golden/make_golden_ref_gpu.py [OUT.npz]

Per output: its shape, its abs max, and its values at the SAMPLE positions of test_ref_gpu.sample_positions (all
of them when it is no larger); per input: its first PROBE values, so that a drift of the seeded generators shows
as such.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, TESTS)
sys.path.insert(0, os.path.dirname(TESTS))

import test_ref_gpu as T  # noqa: E402
from oracle import ref_gpu  # noqa: E402


def main(path):
    assert ref_gpu.available(), "oracle/_ref/libdcnv2_ref.so is not built"
    out = {}

    def inputs(k, *tensors):
        for i, t in enumerate(tensors):
            if t is not None:
                out["%s__in%d" % (k, i)] = t.detach().reshape(-1)[:T.PROBE].cpu().numpy()

    def output(k, t):
        a = t.detach().float().cpu().numpy()
        assert np.isfinite(a).all(), k
        out[k + "__shape"] = np.array(a.shape, np.int64)
        out[k + "__val"] = a.reshape(-1)[T.sample_positions(a.size)]
        out[k + "__absmax"] = np.float64(np.abs(a).max())

    cuda = lambda ts: [t.cuda() for t in ts]  # noqa: E731

    x, off, m, w, b = T.kat_inputs()
    inputs("kat", x)
    output("kat", ref_gpu.dcn_v2_forward(*cuda((x, off, m, w, b))))

    for cfg in T.LAYERS:
        B, Ci, H, W, Co, dg, stride = cfg
        k = T.key("fwd", cfg)
        ins = T.make(*cfg)
        inputs(k, *ins)
        output(k, ref_gpu.dcn_v2_forward(*cuda(ins), stride, 1, 1, dg))

    for cfg in T.FP32_LAYERS:
        B, Ci, H, W, Co, dg, stride = cfg
        k = T.key("fp32", cfg)
        ins = T.make(*cfg, seed=5)
        inputs(k, *ins)
        output(k, ref_gpu.dcn_v2_forward(*cuda(ins), stride, 1, 1, dg))

    for cfg in T.BWD_LAYERS:
        B, Ci, H, W, Co, dg, stride = cfg
        k = T.key("bwd", cfg)
        ins, go = T.bwd_inputs(*cfg)
        inputs(k, *ins, go)
        grads = ref_gpu.dcn_v2_backward(*cuda(ins), go.cuda(), stride, 1, 1, dg)
        for name, g in zip(T.GRADS, grads):
            output(k + "_" + name, g)

    for case in T.PS_CASES:
        k = "psroi_%d" % case[0]
        data, rois, trans, cfg = T._case(*case)
        inputs(k, torch.from_numpy(data), torch.from_numpy(rois), None if trans is None else torch.from_numpy(trans))
        d = torch.from_numpy(data).cuda(); r = torch.from_numpy(rois).cuda()
        t = torch.zeros(1, device="cuda") if trans is None else torch.from_numpy(trans).cuda()
        kw = T.psroi_kwargs(cfg)
        ref_out, ref_cnt = ref_gpu.psroi_forward(d, r, t, **kw)
        go = torch.from_numpy(T.psroi_grad_out(ref_out.shape)).cuda()
        ref_gi, ref_gt = ref_gpu.psroi_backward(go, d, r, t, ref_cnt, **kw)
        output(k + "_out", ref_out)
        output(k + "_cnt", ref_cnt)
        output(k + "_gi", ref_gi)
        if trans is not None:
            output(k + "_gt", ref_gt)

    torch.cuda.synchronize()
    np.savez_compressed(path, **out)
    print("wrote %s: %d arrays, %d bytes on %s" % (path, len(out), os.path.getsize(path),
                                                   torch.cuda.get_device_name(0)))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "ref_gpu.npz"))
