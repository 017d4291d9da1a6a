"""CPU oracle for the box-op half of the hot path (numpy, float32, op-by-op).

TEST INFRASTRUCTURE ONLY.  Nothing under ``ssds_pytorch_b200/`` may import this
module; only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs use it, and only as the checker or
as the timed CPU baseline.

It restates, in plain numpy, the algorithms of the reference's
``ssds/modeling/layers/box.py``, ``ssds/modeling/layers/decoder.py`` and
``ssds/core/criterion.py`` (reference @ b5ec682).  Every function cites the
reference lines it follows.  Arithmetic is kept in float32 and in the same
operation order as the reference's torch expressions, so +,-,*,/ and sqrt are
bit-identical to the torch CPU path; exp/log may differ by an ulp.

Parity pinning: the reference ships no golden vectors (SURVEY.md section 4), so this
oracle is pinned against *outputs of the reference itself*, generated in the
authoring container by ``tests/golden/make_golden.py`` (imports
``/root/reference``) and committed under ``tests/golden/*.npz``;
``tests/test_oracle_golden.py`` replays them.

Where the reference leaves an order implementation-defined the oracle fixes
the rule the CUDA kernels implement:
  * ``torch.topk`` / ``torch.sort`` ties  -> descending score, ascending flat
    index among equals (a stable descending sort; matches torch CPU ``sort``).
  * ``Tensor.max(dim)`` ties              -> first maximum (matches torch CPU).
"""
import numpy as np

f32 = np.float32


# --------------------------------------------------------------------------- #
# anchors ("PriorBox")
# --------------------------------------------------------------------------- #
def generate_anchors(stride, ratio_vals, scales_vals):
    """Base anchors [A,4] — reference box.py:46-58.

    Order is scale-major, ratio-minor (box.py:49-51).  ``torch.round`` is
    round-half-to-even (np.rint), which matters e.g. for stride 15 / ratio 0.5.
    """
    scales = np.repeat(np.asarray(scales_vals, dtype=f32), len(ratio_vals)).reshape(-1, 1)
    ratios = np.asarray(list(ratio_vals) * len(scales_vals), dtype=f32)
    wh = np.full((len(ratios), 2), stride, dtype=f32)
    ws = np.rint(np.sqrt(wh[:, 0] * wh[:, 1] / ratios)).astype(f32)
    dwh = np.stack([ws, np.rint(ws * ratios).astype(f32)], axis=1)
    xy1 = f32(0.5) * (wh - dwh * scales)
    xy2 = f32(0.5) * (wh + dwh * scales) - f32(1)
    return np.concatenate([xy1, xy2], axis=1).astype(f32)


def anchor_grid(base, stride, width, height):
    """Materialised anchor grid in the reference's order [A, W, H, 4] (x-major!).

    reference box.py:151-159 (``meshgrid`` with ij semantics on (x, y)).
    """
    x = np.arange(0, width * stride, stride, dtype=f32)
    y = np.arange(0, height * stride, stride, dtype=f32)
    xx, yy = np.meshgrid(x, y, indexing="ij")           # [W,H]
    xyxy = np.stack((xx, yy, xx, yy), axis=2)[None]     # [1,W,H,4]
    return (xyxy + base.reshape(-1, 1, 1, 4).astype(f32)).astype(f32)


# --------------------------------------------------------------------------- #
# encode / decode of boxes
# --------------------------------------------------------------------------- #
def box2delta(boxes, anchors):
    """reference box.py:61-71 ("encode")."""
    boxes = boxes.astype(f32)
    anchors = anchors.astype(f32)
    anchors_wh = anchors[:, 2:] - anchors[:, :2] + f32(1)
    anchors_ctr = anchors[:, :2] + f32(0.5) * anchors_wh
    boxes_wh = boxes[:, 2:] - boxes[:, :2] + f32(1)
    boxes_ctr = boxes[:, :2] + f32(0.5) * boxes_wh
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.concatenate(
            [(boxes_ctr - anchors_ctr) / anchors_wh, np.log(boxes_wh / anchors_wh)], axis=1
        ).astype(f32)


def delta2box(deltas, anchors, size, stride):
    """reference box.py:74-87 ("decode (box)"); ``size`` = [W_feat, H_feat]."""
    deltas = deltas.astype(f32)
    anchors = anchors.astype(f32)
    anchors_wh = anchors[:, 2:] - anchors[:, :2] + f32(1)
    ctr = anchors[:, :2] + f32(0.5) * anchors_wh
    pred_ctr = deltas[:, :2] * anchors_wh + ctr
    with np.errstate(over="ignore"):
        pred_wh = np.exp(deltas[:, 2:]).astype(f32) * anchors_wh
    m = np.zeros([2], dtype=f32)
    M = np.asarray(size, dtype=f32) * f32(stride) - f32(1)

    def clamp(t):
        # torch.max(m, torch.min(t, M)) propagates NaN
        return np.maximum(m, np.minimum(t, M))

    return np.concatenate(
        [clamp(pred_ctr - f32(0.5) * pred_wh), clamp(pred_ctr + f32(0.5) * pred_wh - f32(1))],
        axis=1,
    ).astype(f32)


# --------------------------------------------------------------------------- #
# decode (threshold + top-k + box + centerness rescore)
# --------------------------------------------------------------------------- #
def topk_desc_stable(values, k):
    """Indices of the k largest, descending, ascending index among equals."""
    order = np.argsort(-values.astype(np.float64), kind="stable")
    return order[:k]


def decode(all_cls_head, all_box_head, stride=1, threshold=0.05, top_n=1000,
           anchors=None, rescore=True, return_indices=False):
    """reference box.py:408-477.

    all_cls_head [B, A*C, H, W] (already sigmoid-ed), all_box_head [B, A*4, H, W],
    anchors [A,4].  Returns zero-padded scores [B,top_n], boxes [B,top_n,4],
    classes [B,top_n] (float32, like the reference), and optionally the flat
    indices [B,top_n] (int64, -1 padded) of the kept scores.
    """
    all_cls_head = np.asarray(all_cls_head, dtype=f32)
    all_box_head = np.asarray(all_box_head, dtype=f32)
    anchors = np.asarray(anchors, dtype=f32)
    num_anchors = anchors.shape[0]
    num_classes = all_cls_head.shape[1] // num_anchors
    height, width = all_cls_head.shape[-2:]
    batch_size = all_cls_head.shape[0]
    out_scores = np.zeros((batch_size, top_n), dtype=f32)
    out_boxes = np.zeros((batch_size, top_n, 4), dtype=f32)
    out_classes = np.zeros((batch_size, top_n), dtype=f32)
    out_idx = np.full((batch_size, top_n), -1, dtype=np.int64)
    thr = f32(threshold)

    for b in range(batch_size):
        cls_head = all_cls_head[b].reshape(-1)
        box_head = all_box_head[b].reshape(num_anchors, 4, height, width)
        keep = np.nonzero(cls_head >= thr)[0]                     # box.py:440
        if keep.size == 0:
            continue
        scores = cls_head[keep]
        sel = topk_desc_stable(scores, min(top_n, keep.size))     # box.py:446
        scores = scores[sel]
        indices = keep[sel]
        classes = ((indices // width // height) % num_classes).astype(f32)   # box.py:448
        x = indices % width
        y = (indices // width) % height
        a = indices // num_classes // height // width
        boxes = box_head[a, :, y, x]
        grid = np.stack([x, y, x, y], axis=1).astype(f32) * f32(stride) + anchors[a, :]
        boxes = delta2box(boxes, grid, [width, height], stride)
        if rescore:                                               # box.py:464-471
            grid_center = (grid[:, :2] + grid[:, 2:]) / f32(2)
            lt = np.abs(grid_center - boxes[:, :2])
            rb = np.abs(boxes[:, 2:] - grid_center)
            with np.errstate(divide="ignore", invalid="ignore"):
                q = np.minimum(lt, rb) / np.maximum(lt, rb)
                centerness = np.sqrt(q[:, 0] * q[:, 1]).astype(f32)
            scores = scores * centerness
        n = scores.shape[0]
        out_scores[b, :n] = scores
        out_boxes[b, :n] = boxes
        out_classes[b, :n] = classes
        out_idx[b, :n] = indices
    if return_indices:
        return out_scores, out_boxes, out_classes, out_idx
    return out_scores, out_boxes, out_classes


# --------------------------------------------------------------------------- #
# NMS
# --------------------------------------------------------------------------- #
def nms(all_scores, all_boxes, all_classes, nms=0.5, ndetections=100, using_diou=True,
        return_indices=False):
    """reference box.py:480-546, including its compaction loop.

    Class-aware, +1 pixel areas, 1e-7 eps, DIoU on *top-left corners* (box.py:527).
    ``return_indices`` adds the position of each kept box in the input row
    ([B,ndetections] int64, -1 padded) — an output the reference does not have.
    """
    all_scores = np.asarray(all_scores, dtype=f32)
    all_boxes = np.asarray(all_boxes, dtype=f32)
    all_classes = np.asarray(all_classes, dtype=f32)
    batch_size = all_scores.shape[0]
    out_scores = np.zeros((batch_size, ndetections), dtype=f32)
    out_boxes = np.zeros((batch_size, ndetections, 4), dtype=f32)
    out_classes = np.zeros((batch_size, ndetections), dtype=f32)
    out_idx = np.full((batch_size, ndetections), -1, dtype=np.int64)
    thr = f32(nms)
    eps = f32(1e-7)

    for b in range(batch_size):
        keep = np.nonzero(all_scores[b].reshape(-1) > 0)[0]        # box.py:496 (NaN dropped)
        if keep.size == 0:
            continue
        scores = all_scores[b, keep]
        boxes = all_boxes[b, keep, :].reshape(-1, 4)
        classes = all_classes[b, keep]
        order = np.argsort(-scores.astype(np.float64), kind="stable")   # box.py:505
        scores, boxes, classes, orig = scores[order], boxes[order], classes[order], keep[order]
        areas = (boxes[:, 2] - boxes[:, 0] + f32(1)) * (boxes[:, 3] - boxes[:, 1] + f32(1))
        i = -1
        broke = False
        for i in range(ndetections):
            if i >= scores.shape[0]:                               # box.py:513-515
                i -= 1
                broke = True
                break
            xy1 = np.maximum(boxes[:, :2], boxes[i, :2])
            xy2 = np.minimum(boxes[:, 2:], boxes[i, 2:])
            wh = np.maximum(xy2 - xy1 + f32(1), f32(0))
            inter = wh[:, 0] * wh[:, 1]
            with np.errstate(divide="ignore", invalid="ignore"):
                iou = inter / (areas + areas[i] - inter + eps)
                if using_diou:
                    outer_lt = np.minimum(boxes[:, :2], boxes[i, :2])
                    outer_rb = np.maximum(boxes[:, 2:], boxes[i, 2:])
                    d = boxes[:, :2] - boxes[i, :2]
                    inter_diag = d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]
                    o = outer_rb - outer_lt
                    outer_diag = (o[:, 0] * o[:, 0] + o[:, 1] * o[:, 1]) + eps
                    iou = np.clip(iou - inter_diag / outer_diag, f32(-1.0), f32(1.0))
                criterion = (scores > scores[i]) | (iou <= thr) | (classes != classes[i])
            criterion[i] = True
            scores, boxes, classes = scores[criterion], boxes[criterion], classes[criterion]
            areas, orig = areas[criterion], orig[criterion]
        n = i + 1
        out_scores[b, :n] = scores[:n]
        out_boxes[b, :n] = boxes[:n]
        out_classes[b, :n] = classes[:n]
        out_idx[b, :n] = orig[:n]
    if return_indices:
        return out_scores, out_boxes, out_classes, out_idx
    return out_scores, out_boxes, out_classes


def decoder_call(loc, conf, anchors, conf_threshold, nms_threshold, top_n, top_n_per_level,
                 rescore, use_diou):
    """reference decoder.py:25-49 — per-level decode, concat along dim 1, nms.

    ``anchors`` is an ordered mapping {stride: base_anchors[A,4]}.
    """
    decoded = [
        decode(c, l, stride, conf_threshold, top_n_per_level, anchor, rescore)
        for l, c, (stride, anchor) in zip(loc, conf, anchors.items())
    ]
    decoded = [np.concatenate(t, axis=1) for t in zip(*decoded)]
    return nms(*decoded, nms=nms_threshold, ndetections=top_n, using_diou=use_diou)


def mean_average_precision(detections, targets, num_classes, conf_threshold, iou_threshold):
    """reference evaluation_metrics.py:5-142 — ``detections`` = (scores [B,D], boxes [B,D,4], classes [B,D]),
    ``targets`` = per image [T,5] (x1, y1, x2, y2, class).  Per image and class, each detection above
    conf_threshold takes the target it overlaps most and is a true positive if that IoU reaches iou_threshold and
    the target is still free.  AP per class is the area under the precision/recall curve with precision made
    non-increasing (VOC all-point); classes without targets are NaN and left out of the mean."""
    hits = [([], []) for _ in range(num_classes)]
    npos = np.zeros(num_classes, np.int64)
    for s, b, c, t in zip(*(np.asarray(a) for a in detections), targets):
        t = np.asarray(t, np.float32)
        keep = s > conf_threshold
        s, b, c = s[keep], b[keep].astype(np.float32), c[keep]
        for k in range(num_classes):
            tk, sk, bk = t[t[:, 4] == k, :4], s[c == k], b[c == k]
            npos[k] += len(tk)
            tp = np.zeros(len(sk), bool)
            if len(sk) and len(tk):
                lt = np.maximum(bk[:, None, :2], tk[:, :2])
                rb = np.minimum(bk[:, None, 2:], tk[:, 2:])
                inter = np.prod(rb - lt, axis=2) * (lt < rb).all(axis=2)
                area_b = np.prod(bk[:, 2:] - bk[:, :2], axis=1)
                area_t = np.prod(tk[:, 2:] - tk[:, :2], axis=1)
                iou = inter / (area_b[:, None] + area_t - inter)
                taken = np.zeros(len(tk), bool)
                for i, j in enumerate(iou.argmax(axis=1)):
                    if iou[i, j] >= iou_threshold and not taken[j]:
                        taken[j] = tp[i] = True
            hits[k][0].extend(sk.tolist())
            hits[k][1].extend(tp.tolist())
    aps = []
    for k in range(num_classes):
        if npos[k] == 0:
            aps.append(np.nan)
            continue
        order = np.argsort(np.asarray(hits[k][0], np.float64))[::-1]
        tp = np.asarray(hits[k][1], np.int64)[order]
        ctp, cfp = np.cumsum(tp), np.cumsum(1 - tp)
        rec = np.concatenate([[0], ctp / float(npos[k]), [1]])
        prec = np.concatenate([[0], ctp / np.maximum(ctp + cfp, np.finfo(np.float64).eps), [0]])
        prec = np.maximum.accumulate(prec[::-1])[::-1]
        step = np.nonzero(rec[1:] != rec[:-1])[0] + 1
        aps.append(np.sum((rec[step] - rec[step - 1]) * prec[step]))
    return float(np.nanmean(aps))


# --------------------------------------------------------------------------- #
# match ("jaccard" + "match" + "encode")
# --------------------------------------------------------------------------- #
def snap_to_anchors_by_iou(boxes, size, stride, anchors, num_classes, match,
                           center_sampling_radius=0):
    """reference box.py:116-226 (is_centerness=False path).

    boxes [T,5] = (x, y, w, h, label) with padded rows already removed;
    ``size`` = [W_img, H_img] (= feature size * stride).  Returns
    cls_target [A,C,H,W], box_target [A,4,H,W], depth [A,1,H,W].
    """
    anchors = np.asarray(anchors, dtype=f32)
    num_anchors = anchors.shape[0]
    width, height = int(size[0] / stride), int(size[1] / stride)
    if boxes.size == 0:                                            # box.py:132-145
        return (np.zeros([num_anchors, num_classes, height, width], f32),
                np.zeros([num_anchors, 4, height, width], f32),
                np.zeros([num_anchors, 1, height, width], f32))
    boxes = np.asarray(boxes, dtype=f32)
    boxes, classes = boxes[:, :4], boxes[:, 4:]
    match_threshold, unmatch_threshold = f32(match[0]), f32(match[1])

    grid = anchor_grid(anchors, stride, width, height).reshape(-1, 4)   # [A*W*H,4]

    boxes = np.concatenate([boxes[:, :2], boxes[:, :2] + boxes[:, 2:] - f32(1)], axis=1)
    xy1 = np.maximum(grid[:, None, :2], boxes[:, :2])
    xy2 = np.minimum(grid[:, None, 2:], boxes[:, 2:])
    wh = np.maximum(xy2 - xy1 + f32(1), f32(0))
    inter = wh[..., 0] * wh[..., 1]
    b_wh = boxes[:, 2:] - boxes[:, :2] + f32(1)
    boxes_area = b_wh[:, 0] * b_wh[:, 1]
    a_wh = grid[:, 2:] - grid[:, :2] + f32(1)
    anchors_area = a_wh[:, 0] * a_wh[:, 1]
    with np.errstate(divide="ignore", invalid="ignore"):
        overlap = inter / (anchors_area[:, None] + boxes_area - inter)

    indices = np.argmax(overlap, axis=1)                           # first max, box.py:171
    overlap = overlap[np.arange(overlap.shape[0]), indices]
    box_target = box2delta(boxes[indices], grid)
    box_target = box_target.reshape(num_anchors, width, height, 4).transpose(0, 3, 2, 1)

    depth = np.full_like(overlap, -1, dtype=f32)
    depth[overlap < unmatch_threshold] = 0
    pos = overlap >= match_threshold
    depth[pos] = classes[indices][pos].reshape(-1) + f32(1)
    depth = depth.reshape(num_anchors, width, height)
    if center_sampling_radius > 0:                                 # box.py:184-191, 90-113
        xg = np.arange(0, width * stride, stride, dtype=f32)
        yg = np.arange(0, height * stride, stride, dtype=f32)
        xx, yy = np.meshgrid(xg, yg, indexing="ij")
        pts = np.stack((xx, yy), axis=2) + f32(stride // 2)        # [W,H,2]
        r = f32(stride * center_sampling_radius)
        center = (boxes[:, :2] + boxes[:, 2:]) / f32(2)
        cb = np.concatenate((center - r, center + r), axis=-1)
        lt = pts[:, :, None, :] - np.maximum(cb[:, :2], boxes[:, :2])[None, None]
        rb = np.minimum(cb[:, 2:], boxes[:, 2:])[None, None] - pts[:, :, None, :]
        inside = (np.concatenate((lt, rb), -1).min(-1) > 0).astype(f32).max(-1)   # [W,H]
        depth = np.minimum(depth, inside[None])
    depth = depth.transpose(0, 2, 1)

    cls_idx = classes[indices].reshape(-1).astype(np.int64)
    cls_idx[overlap < unmatch_threshold] = num_classes             # background: dropped column
    cls_target = np.zeros((grid.shape[0], num_classes + 1), dtype=f32)
    cls_target[np.arange(grid.shape[0]), cls_idx] = 1
    cls_target = cls_target[:, :num_classes].reshape(num_anchors, width, height, num_classes)
    cls_target = cls_target.transpose(0, 3, 2, 1)
    return (np.ascontiguousarray(cls_target, dtype=f32),
            np.ascontiguousarray(box_target, dtype=f32),
            np.ascontiguousarray(depth.reshape(num_anchors, 1, height, width), dtype=f32))


def extract_targets(targets, anchors, classes, stride, size, match=(0.5, 0.4),
                    center_sampling_radius=0):
    """reference box.py:362-405 (IoU matcher only; ``match[0]`` must be a float).

    targets [B,T,5] padded with -1 rows; ``size`` = (H_feat, W_feat).
    """
    if not isinstance(match[0], float):
        raise ValueError("unvalidate match param")                 # box.py:402
    cls_t, box_t, dep = [], [], []
    for target in np.asarray(targets, dtype=f32):
        target = target[target[:, -1] > -1]                        # box.py:375
        s = snap_to_anchors_by_iou(target, [v * stride for v in size[::-1]], stride,
                                   anchors[stride], classes, match, center_sampling_radius)
        cls_t.append(s[0]); box_t.append(s[1]); dep.append(s[2])
    return np.stack(cls_t), np.stack(box_t), np.stack(dep)


# --------------------------------------------------------------------------- #
# MultiBoxLoss
# --------------------------------------------------------------------------- #
def bce_with_logits(x, t):
    """torch F.binary_cross_entropy_with_logits, reduction='none':
    (1 - t) * x - log_sigmoid(x), log_sigmoid(x) = min(x,0) - log1p(exp(-|x|))."""
    x = x.astype(f32)
    t = t.astype(f32)
    ls = np.minimum(x, f32(0)) - np.log1p(np.exp(-np.abs(x))).astype(f32)
    return ((f32(1) - t) * x - ls).astype(f32)


def multibox_loss(pred_logits, target, depth, negpos_ratio=3):
    """reference criterion.py:43-71 with the intended per-image semantics.

    The reference's ``num_neg.expand_as`` (criterion.py:66-68) only runs for
    B == 1; the intended meaning (``num_neg[:, None]``) is applied per image, which
    is exactly what calling the reference on B=1 slices gives (SURVEY 8a-7).
    Rank ties follow a stable descending sort (lower flat index ranks first).
    pred_logits/target [B,A,C,H,W], depth [B,A,1,H,W]; returns unreduced [B,A,C,H,W].
    """
    pred_logits = np.asarray(pred_logits, dtype=f32)
    target = np.asarray(target, dtype=f32)
    depth = np.asarray(depth, dtype=f32)
    ce = bce_with_logits(pred_logits, target)
    B = ce.shape[0]
    out = np.zeros_like(ce)
    for b in range(B):
        max_ce = ce[b].max(axis=1).reshape(-1).copy()              # over C -> [A*H*W]
        depth_v = depth[b].reshape(-1)
        max_ce[depth_v != 0] = 0
        idx = np.argsort(-max_ce.astype(np.float64), kind="stable")
        rank = np.empty_like(idx)
        rank[idx] = np.arange(idx.size)
        num_pos = int((depth_v > 0).sum())
        num_neg = min(negpos_ratio * num_pos, depth_v.size - 1)
        neg = (rank < num_neg).reshape(depth[b].shape)
        mask = ((depth[b] > 0) | neg)
        out[b] = ce[b] * mask.astype(f32)
    return out


def multibox_loss_reduced(pred_logits, target, depth, negpos_ratio=3):
    """Caller-side reduction, reference pipeline_anchor_basic.py:76-82:
    per image (sum of loss * (depth >= 0), count of depth > 0)."""
    loss = multibox_loss(pred_logits, target, depth, negpos_ratio)
    depth = np.asarray(depth, dtype=f32)
    B = loss.shape[0]
    m = (depth >= 0).astype(f32)
    sums = (loss * m).reshape(B, -1).astype(np.float64).sum(axis=1)
    npos = (depth > 0).reshape(B, -1).sum(axis=1)
    return sums, npos


# --------------------------------------------------------------------------- #
# Focal / SmoothL1 / IoU-family losses (SURVEY 8f rank 1)
# --------------------------------------------------------------------------- #
def focal_loss(pred_logits, target, alpha=0.25, gamma=2):
    """reference criterion.py:95-108 — alpha_t * (1 - p_t)^gamma * BCEWithLogits, unreduced."""
    x = np.asarray(pred_logits, dtype=f32)
    t = np.asarray(target, dtype=f32)
    p = (f32(1) / (f32(1) + np.exp(-x).astype(f32))).astype(f32)
    ce = bce_with_logits(x, t)
    a = (t * f32(alpha) + (f32(1) - t) * f32(1 - alpha)).astype(f32)
    pt = np.where(t == 1, p, f32(1) - p).astype(f32)
    return (a * (f32(1) - pt) ** f32(gamma) * ce).astype(f32)


def smooth_l1_loss(pred, target, beta=0.11):
    """reference criterion.py:138-151."""
    x = np.abs(np.asarray(pred, dtype=f32) - np.asarray(target, dtype=f32)).astype(f32)
    b = f32(beta)
    return np.where(x >= b, x - f32(0.5) * b, f32(0.5) * x * x / b).astype(f32)


def _delta2ltrb(d):
    """reference criterion.py:233-239: [B,A,4,H,W] (x, y, log w, log h) -> ltrb."""
    ctr = d[:, :, :2]
    wh = np.exp(d[:, :, 2:]).astype(f32)
    return np.concatenate([ctr - f32(0.5) * wh, ctr + f32(0.5) * wh], axis=2).astype(f32)


def iou_loss(pred, target, loss_type="iou"):
    """reference criterion.py:175-231; pred/target [B,A,4,H,W] deltas -> [B,A,1,H,W]."""
    pred = np.asarray(pred, dtype=f32)
    target = np.asarray(target, dtype=f32)
    p, t = _delta2ltrb(pred), _delta2ltrb(target)
    eps = f32(1e-7)

    def area(lt, rb):
        en = (lt < rb).all(axis=2).astype(f32)
        return ((rb - lt).prod(axis=2) * en).astype(f32)

    lt = np.maximum(p[:, :, :2], t[:, :, :2])
    rb = np.minimum(p[:, :, 2:], t[:, :, 2:])
    area_i = area(lt, rb)
    area_a = np.exp(pred[:, :, 2:]).astype(f32).prod(axis=2).astype(f32)       # prod(pred_wh), :188
    area_b = np.exp(target[:, :, 2:]).astype(f32).prod(axis=2).astype(f32)
    area_u = (area_a + area_b - area_i).astype(f32)
    iou = ((area_i + eps) / (area_u + eps)).astype(f32)
    if loss_type == "iou":
        return (f32(1) - np.clip(iou, 0, 1))[:, :, None].astype(f32)
    olt = np.minimum(p[:, :, :2], t[:, :, :2])
    orb = np.maximum(p[:, :, 2:], t[:, :, 2:])
    if loss_type == "giou":
        area_o = (area(olt, orb) + eps).astype(f32)
        g = (iou - (area_o - area_u) / area_o).astype(f32)
        return (f32(1) - np.clip(g, -1, 1))[:, :, None].astype(f32)
    inter_diag = ((pred[:, :, :2] - target[:, :, :2]) ** 2).sum(axis=2).astype(f32)
    outer_diag = (((orb - olt) ** 2).sum(axis=2) + eps).astype(f32)
    if loss_type == "diou":
        d = (iou - inter_diag / outer_diag).astype(f32)
        return (f32(1) - np.clip(d, -1, 1))[:, :, None].astype(f32)
    if loss_type == "ciou":
        pw, ph = np.exp(pred[:, :, 2]).astype(f32), np.exp(pred[:, :, 3]).astype(f32)
        tw, th = np.exp(target[:, :, 2]).astype(f32), np.exp(target[:, :, 3]).astype(f32)
        v = (f32(4 / (np.pi ** 2)) * (np.arctan(tw / th).astype(f32) - np.arctan(pw / ph).astype(f32)) ** 2)
        v = v.astype(f32)
        S = f32(1) - iou
        al = (v / (S + v)).astype(f32)
        c = (iou - (inter_diag / outer_diag + al * v)).astype(f32)
        return (f32(1) - np.clip(c, -1, 1))[:, :, None].astype(f32)
    raise ValueError(loss_type)


def assert_iou_loss_close(got, ref, pred, target, rtol=1e-5, atol=2e-6, msg=""):
    """Comparison helper for the IoU family.  For IDENTICAL pred/target boxes the reference's ciou is
    alpha = v / (1 - iou + v) with v == 0 and 1 - iou either exactly 0 (-> NaN) or one ulp (-> loss ~1e-7),
    depending on the exp() implementation's last bit: that corner is ill-conditioned in the reference
    itself, so there each side only has to be NaN or ~0; everywhere else values (and finiteness) must agree."""
    same = (np.asarray(pred) == np.asarray(target)).all(axis=2, keepdims=True)
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape == same.shape, (got.shape, ref.shape, same.shape)
    np.testing.assert_allclose(got[~same], ref[~same], rtol=rtol, atol=atol, err_msg=msg)
    for v in (got[same], ref[same]):
        assert (np.isnan(v) | (np.abs(v) < 1e-5)).all(), msg


def loc_loss(pred, target, loss_type="smoothl1", beta=0.11):
    return smooth_l1_loss(pred, target, beta) if loss_type == "smoothl1" else iou_loss(pred, target, loss_type)


def masked_loss_sums(cls_loss, loc_loss_v, depth):
    """Caller-side reduction, pipeline_anchor_basic.py:76-97: per image
    (sum(cls * (depth >= 0)), sum(loc * (depth > 0)), #fg)."""
    depth = np.asarray(depth, dtype=f32)
    B = depth.shape[0]
    cs = (cls_loss * (depth >= 0)).reshape(B, -1).astype(np.float64).sum(axis=1)
    ls = (loc_loss_v * (depth > 0)).reshape(B, -1).astype(np.float64).sum(axis=1)
    return cs, ls, (depth > 0).reshape(B, -1).sum(axis=1)
