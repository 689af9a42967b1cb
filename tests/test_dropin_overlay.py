"""A17 / drop-in boundary: dropin/ overlaid on a temp copy of the reference's src/ -- the reference's own
callers (detectors/*.py, trains/*.py, models/model.py, the DCN networks) import and build unchanged on top
of centernet_b200.  CPU; needs a checkout of the original CenterNet, whose src/ directory CENTERNET_SRC names
(skipped without it).  The run happens in a subprocess so the stub modules and sys.path edits stay out of the
test process."""
import os
import shutil
import subprocess
import sys
import textwrap

import pytest

REF_SRC = os.environ.get("CENTERNET_SRC", "")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCRIPT = textwrap.dedent('''
    import sys, types, os
    src = sys.argv[1]
    # stubs for the packages this image lacks (SURVEY 8c): progress, matplotlib, pycocotools
    def stub(name, **attrs):
        m = types.ModuleType(name); m.__dict__.update(attrs); sys.modules[name] = m; return m
    class Bar(object):
        def __init__(self, *a, **k): pass
        def next(self): pass
        def finish(self): pass
    stub("progress"); stub("progress.bar", Bar=Bar)
    stub("matplotlib"); stub("matplotlib.pyplot"); stub("mpl_toolkits"); stub("mpl_toolkits.mplot3d", Axes3D=object)
    stub("pycocotools"); stub("pycocotools.coco", COCO=object); stub("pycocotools.cocoeval", COCOeval=object)
    sys.path.insert(0, os.path.join(src, "lib")); sys.path.insert(0, src)
    import torch
    import centernet_b200
    from centernet_b200 import decode as D, utils as U, losses as L, dcn_v2 as DC

    import models.decode, models.utils, models.losses
    for name in ("_nms", "_topk", "_topk_channel", "ctdet_decode", "multi_pose_decode", "exct_decode",
                 "agnex_ct_decode", "ddd_decode", "_h_aggregate", "_v_aggregate"):
        assert getattr(models.decode, name) is getattr(D, name), name
    for name in ("_sigmoid", "_gather_feat", "_transpose_and_gather_feat", "flip_tensor", "flip_lr", "flip_lr_off"):
        assert getattr(models.utils, name) is getattr(U, name), name
    for name in ("FocalLoss", "RegL1Loss", "RegLoss", "NormRegL1Loss", "RegWeightedL1Loss", "L1Loss", "BinRotLoss"):
        assert getattr(models.losses, name) is getattr(L, name), name

    import utils.post_process, external.nms, models.data_parallel
    from centernet_b200 import post_process as PP, data_parallel as DP
    assert utils.post_process.ctdet_post_process is PP.ctdet_post_process
    assert utils.post_process.multi_pose_post_process is PP.multi_pose_post_process
    assert callable(utils.post_process.ddd_post_process)            # served by the untouched reference code
    assert external.nms.soft_nms is PP.soft_nms and external.nms.soft_nms_39 is PP.soft_nms_39
    assert models.data_parallel.DataParallel is DP.DataParallel

    from detectors.detector_factory import detector_factory
    assert set(detector_factory) == {"exdet", "ddd", "ctdet", "multi_pose"}
    import detectors.ctdet, detectors.multi_pose, detectors.exdet
    assert detectors.ctdet.ctdet_decode is D.ctdet_decode
    assert detectors.multi_pose.multi_pose_decode is D.multi_pose_decode
    assert detectors.exdet.exct_decode is D.exct_decode
    from trains.train_factory import train_factory
    assert set(train_factory) == {"exdet", "ddd", "ctdet", "multi_pose"}
    import trains.ctdet, trains.base_trainer
    assert trains.ctdet.FocalLoss is L.FocalLoss and trains.ctdet.ctdet_decode is D.ctdet_decode
    assert trains.base_trainer.DataParallel is DP.DataParallel
    assert detectors.ctdet.ctdet_post_process is PP.ctdet_post_process and detectors.ctdet.soft_nms is PP.soft_nms

    # the DCN networks build on the overlaid DCNv2 package (pose_dla_dcn.py:16, resnet_dcn.py:18)
    from models.networks import pose_dla_dcn
    pose_dla_dcn.DLA.load_pretrained_model = lambda self, *a, **k: None      # no network
    from models.model import create_model
    heads = {"hm": 80, "wh": 2, "reg": 2}
    net = create_model("dla_34", heads, 256)
    dcns = [m for m in net.modules() if isinstance(m, DC.DCN)]
    assert len(dcns) == 16, len(dcns)
    keys = net.state_dict().keys()
    assert any(k.endswith("conv_offset_mask.weight") for k in keys)
    import torch.utils.model_zoo as zoo
    zoo.load_url = lambda *a, **k: {}
    net2 = create_model("resdcn_18", heads, 64)
    assert sum(isinstance(m, DC.DCN) for m in net2.modules()) == 3

    # opts surface unchanged
    from opts import opts
    opt = opts().init("ctdet --arch dla_34 --gpus -1".split(" "))
    assert opt.heads == {"hm": 80, "wh": 2, "reg": 2} and opt.K == 100
    # no CPU fallback: the overlaid op raises exactly like the reference's DCNv2Function (dcn_v2_func.py:23-24)
    try:
        D.ctdet_decode(torch.zeros(1, 2, 8, 8), torch.zeros(1, 2, 8, 8))
    except NotImplementedError:
        pass
    else:
        raise AssertionError("CPU tensors must raise NotImplementedError")
    print("OVERLAY-OK")
''')


@pytest.mark.skipif(not os.path.isdir(REF_SRC), reason="set CENTERNET_SRC to the src/ of a CenterNet checkout")
def test_reference_callers_import_on_the_overlay(tmp_path):
    src = tmp_path / "src"
    shutil.copytree(REF_SRC, src)
    for dirpath, _, files in os.walk(os.path.join(ROOT, "dropin", "src")):
        for f in files:
            rel = os.path.relpath(os.path.join(dirpath, f), os.path.join(ROOT, "dropin", "src"))
            dst = src / rel
            os.chmod(dst.parent, 0o755)
            if dst.exists():
                os.chmod(dst, 0o644)
                if rel.endswith("utils/post_process.py"):      # INTEGRATION.md: the ddd functions stay with the reference
                    shutil.copyfile(dst, str(dst)[:-3] + "_ref.py")
            shutil.copyfile(os.path.join(dirpath, f), dst)
    # the reference's stale cffi extension directory must not be importable by accident
    script = tmp_path / "run.py"
    script.write_text(SCRIPT)
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, str(script), str(src)], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and "OVERLAY-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
