"""numpy restatement of src/lib/models/losses.py + models/utils.py:_sigmoid
(TEST INFRASTRUCTURE).  fp32 element-wise math in the reference's operation order;
reductions are done in float64 and rounded once, which is what a tolerance-based
comparison (rel 1e-5, SURVEY.md section 8d) expects of any summation order."""
import numpy as np

F32 = np.float32


def sigmoid_clamped(x):
    """models/utils.py:8-10 (_sigmoid): clamp(sigmoid(x), 1e-4, 1-1e-4)."""
    x = np.asarray(x, F32)
    y = (F32(1) / (F32(1) + np.exp(-x.astype(np.float64)))).astype(F32)
    return np.clip(y, F32(1e-4), F32(1 - 1e-4))


def neg_loss(pred, gt):
    """models/losses.py:42-67 (_neg_loss).  Returns (loss, num_pos)."""
    pred = np.asarray(pred, F32); gt = np.asarray(gt, F32)
    pos = (gt == 1).astype(F32)
    neg = (gt < 1).astype(F32)
    neg_w = np.power(F32(1) - gt, 4).astype(F32)
    pos_loss = np.log(pred) * np.power(F32(1) - pred, 2) * pos
    neg_loss_ = np.log(F32(1) - pred) * np.power(pred, 2) * neg_w * neg
    num_pos = float(pos.sum(dtype=np.float64))
    ps = float(pos_loss.sum(dtype=np.float64)); ns = float(neg_loss_.sum(dtype=np.float64))
    if num_pos == 0:
        return F32(-ns), num_pos
    return F32(-(ps + ns) / num_pos), num_pos


def neg_loss_grad(pred, gt):
    """d _neg_loss / d pred (analytic; for checking the fused backward)."""
    return _neg_loss_grad64(pred, gt).astype(F32)


def neg_loss_grad_logits(s32, gt):
    """d (_sigmoid + _neg_loss) / d logit in float64.  s32 is the fp32 sigmoid of the logits (what torch's
    sigmoid returns); torch.clamp's backward passes the gradient only where 1e-4 <= s32 <= 1-1e-4 (inclusive)."""
    s32 = np.asarray(s32, F32)
    lo, hi = F32(1e-4), F32(1 - 1e-4)
    s = s32.astype(np.float64)
    chain = np.where((s32 >= lo) & (s32 <= hi), s * (1 - s), 0.0)
    return _neg_loss_grad64(np.clip(s32, lo, hi), gt) * chain


def _neg_loss_grad64(pred, gt):
    pred = np.asarray(pred, np.float64); gt = np.asarray(gt, np.float64)
    pos = (gt == 1); neg = (gt < 1)
    num_pos = pos.sum()
    g = np.zeros_like(pred)
    # d/dp [log(p)(1-p)^2] = (1-p)^2/p - 2(1-p)log(p)
    g[pos] = ((1 - pred) ** 2 / pred - 2 * (1 - pred) * np.log(pred))[pos]
    # d/dp [log(1-p) p^2 w] = w(2p log(1-p) - p^2/(1-p))
    w = (1 - gt) ** 4
    g[neg] = (w * (2 * pred * np.log(1 - pred) - pred ** 2 / (1 - pred)))[neg]
    return -g / (num_pos if num_pos > 0 else 1.0)


def _gather_pred(output, ind):
    """models/utils.py:22-26 on [B,D,H,W] / ind [B,M] -> [B,M,D]."""
    B, D = output.shape[:2]
    flat = np.asarray(output, F32).reshape(B, D, -1)
    return np.take_along_axis(flat, np.asarray(ind, np.int64)[:, None, :].repeat(D, axis=1), axis=2).transpose(0, 2, 1)


def reg_l1_loss(output, mask, ind, target):
    """models/losses.py:139-149 (RegL1Loss)."""
    pred = _gather_pred(output, ind)
    m = np.asarray(mask, F32)[:, :, None] * np.ones_like(pred)
    s = np.abs(pred * m - np.asarray(target, F32) * m).sum(dtype=np.float64)
    return F32(s / (m.sum(dtype=np.float64) + 1e-4))


def reg_loss(output, mask, ind, target):
    """models/losses.py:98-112,123-137 (RegLoss = smooth-L1 / (num + 1e-4))."""
    pred = _gather_pred(output, ind)
    m = np.asarray(mask, F32)
    num = m.sum(dtype=np.float64)
    mm = m[:, :, None] * np.ones_like(pred)
    d = np.abs(pred * mm - np.asarray(target, F32) * mm).astype(np.float64)
    sl1 = np.where(d < 1, 0.5 * d * d, d - 0.5).sum()
    return F32(sl1 / (num + 1e-4))


def norm_reg_l1_loss(output, mask, ind, target):
    """models/losses.py:151-163 (NormRegL1Loss)."""
    pred = _gather_pred(output, ind)
    target = np.asarray(target, F32)
    m = np.asarray(mask, F32)[:, :, None] * np.ones_like(pred)
    pred = pred / (target + F32(1e-4))
    tgt = target * F32(0) + F32(1)
    s = np.abs(pred * m - tgt * m).sum(dtype=np.float64)
    return F32(s / (m.sum(dtype=np.float64) + 1e-4))


def reg_weighted_l1_loss(output, mask, ind, target):
    """models/losses.py:165-175 (RegWeightedL1Loss; mask is float [B,M,D])."""
    pred = _gather_pred(output, ind)
    m = np.asarray(mask, F32)
    s = np.abs(pred * m - np.asarray(target, F32) * m).sum(dtype=np.float64)
    return F32(s / (m.sum(dtype=np.float64) + 1e-4))
