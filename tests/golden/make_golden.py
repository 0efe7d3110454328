"""Generate the committed golden fixtures (tests/golden/*.npz) from the REAL reference.

Needs a detectron2 source checkout (DETECTRON2_REFERENCE) and torchvision:
    DETECTRON2_REFERENCE=<detectron2 checkout> python tests/golden/make_golden.py [fixture ...]
With fixture names (e.g. `compiled_reference`), only those fixtures are rewritten.

Sources of truth used (never our own code):
  * torchvision CPU ops  -- the reference's backend for roi_align / nms / deform_conv2d
    (detectron2/layers/roi_align.py:3,58; nms.py:5-22; deform_conv.py:9,55)
  * oracle/_ref/d2_ref_cpu.so -- the reference CPU csrc compiled in place (oracle/build.py):
    torch.ops.detectron2.{roi_align_rotated_forward,roi_align_rotated_backward,box_iou_rotated,nms_rotated}
  * detectron2/layers/mask_ops.py of the checkout loaded as a stand-alone module
    (paste_masks_in_image, pure torch)
  * detectron2/layers/deform_conv.py of the checkout: the calls its autograd Functions make into `detectron2._C`
Inputs are seeded; both inputs and outputs are stored so the tests need nothing but the .npz.
"""
import importlib.util
import os
import sys

import numpy as np
import torch
import torchvision
from torchvision.ops import boxes as tv_boxes

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ["DETECTRON2_REFERENCE"]
sys.path.insert(0, ROOT)
from oracle import oracle as orc  # noqa: E402  (only for load_reference())

assert orc.load_reference(), "reference CPU csrc must be built (python oracle/build.py)"
D2 = torch.ops.detectron2


def save(name, **arrs):
    out = {}
    for k, v in arrs.items():
        out[k] = v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, {k: tuple(v.shape) for k, v in out.items()})


def rand_rois(g, k, n, wimg, himg, lo=2.0, hi=None):
    hi = hi or min(wimg, himg) * 0.8
    cx = torch.rand(k, generator=g) * wimg
    cy = torch.rand(k, generator=g) * himg
    w = lo + torch.rand(k, generator=g) * (hi - lo)
    h = lo + torch.rand(k, generator=g) * (hi - lo)
    b = torch.randint(0, n, (k,), generator=g).float()
    rois = torch.stack([b, cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1)
    return rois


def gen_roi_align():
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(2, 8, 24, 32, generator=g)
    rois = rand_rois(g, 40, 2, 64, 48)  # image coords, spatial_scale 0.5
    # edge cases: empty box (tests/layers/test_roi_align.py:111-121), box outside the map, huge box, tiny box
    rois[0] = torch.tensor([0, 3.0, 4.0, 5.0, 4.0])
    rois[1] = torch.tensor([1, -40.0, -30.0, -10.0, -5.0])
    rois[2] = torch.tensor([0, -20.0, -20.0, 200.0, 150.0])
    rois[3] = torch.tensor([1, 10.2, 10.3, 10.9, 11.0])
    rois[4] = torch.tensor([1, 60.0, 40.0, 70.0, 55.0])
    cfgs = [(7, 7, 0, True), (7, 7, 2, True), (5, 3, 0, False), (14, 14, 0, True), (2, 2, 3, False)]
    out = {"x": x, "rois": rois, "cfgs": np.asarray([[a, b, c, int(d)] for a, b, c, d in cfgs])}
    for i, (ph, pw, sr, al) in enumerate(cfgs):
        xi = x.clone().requires_grad_(True)
        y = torchvision.ops.roi_align(xi, rois, (ph, pw), 0.5, sr, al)
        go = torch.randn(y.shape, generator=g)
        y.backward(go)
        out[f"y{i}"] = y
        out[f"go{i}"] = go
        out[f"gx{i}"] = xi.grad
    save("roi_align", **out)


def gen_roi_align_rotated():
    g = torch.Generator().manual_seed(4321)
    x = torch.randn(2, 6, 20, 28, generator=g)
    k = 36
    cx = torch.rand(k, generator=g) * 56
    cy = torch.rand(k, generator=g) * 40
    w = 2 + torch.rand(k, generator=g) * 30
    h = 2 + torch.rand(k, generator=g) * 30
    a = (torch.rand(k, generator=g) - 0.5) * 360
    b = torch.randint(0, 2, (k,), generator=g).float()
    rois = torch.stack([b, cx, cy, w, h, a], 1)
    rois[0] = torch.tensor([0, 2.0, 3.0, 0.0, 0.0, 0.0])  # empty (test_roi_align_rotated.py:102-105)
    rois[1] = torch.tensor([1, 28.0, 20.0, 12.0, 8.0, 90.0])
    rois[2] = torch.tensor([1, -30.0, -30.0, 10.0, 10.0, 33.0])  # outside
    cfgs = [(7, 7, 0), (5, 5, 2), (3, 4, 1)]
    out = {"x": x, "rois": rois, "cfgs": np.asarray(cfgs)}
    for i, (ph, pw, sr) in enumerate(cfgs):
        y = D2.roi_align_rotated_forward(x, rois, 0.5, ph, pw, sr)
        go = torch.randn(y.shape, generator=g)
        gx = D2.roi_align_rotated_backward(go, rois, 0.5, ph, pw, 2, 6, 20, 28, sr)
        out[f"y{i}"] = y
        out[f"go{i}"] = go
        out[f"gx{i}"] = gx
    save("roi_align_rotated", **out)


def random_boxes(g, n, size):  # after detectron2/utils/testing.py:42-53
    b = torch.rand(n, 4, generator=g) * (size * 0.5)
    b[:, 2:] += size * 0.5
    return b


def gen_nms():
    g = torch.Generator().manual_seed(99)
    m = 700
    boxes = random_boxes(g, m, 300)
    # clusters of near-duplicates so that many IoUs sit near the thresholds
    boxes[100:200] = boxes[:100] + torch.randn(100, 4, generator=g) * 3
    boxes[200:230] = boxes[:30]  # exact duplicates
    scores = torch.rand(m, generator=g)
    scores[300:340] = scores[260:300]  # score ties
    idxs = torch.randint(0, 6, (m,), generator=g)
    out = {"boxes": boxes, "scores": scores, "idxs": idxs, "thr": np.asarray([0.2, 0.3, 0.5, 0.7, 0.8])}
    for i, t in enumerate([0.2, 0.3, 0.5, 0.7, 0.8]):
        out[f"keep{i}"] = torchvision.ops.nms(boxes, scores, t)
        out[f"bkeep_trick{i}"] = tv_boxes._batched_nms_coordinate_trick(boxes, scores, idxs, t)
        out[f"bkeep_vanilla{i}"] = tv_boxes._batched_nms_vanilla(boxes, scores, idxs, t)
    save("nms", **out)


def rand_rotated(g, n, size, wmax):
    cx = torch.rand(n, generator=g) * size
    cy = torch.rand(n, generator=g) * size
    w = 1 + torch.rand(n, generator=g) * wmax
    h = 1 + torch.rand(n, generator=g) * wmax
    a = (torch.rand(n, generator=g) - 0.5) * 360
    return torch.stack([cx, cy, w, h, a], 1)


def gen_rotated_iou_nms():
    g = torch.Generator().manual_seed(7)
    b1 = rand_rotated(g, 90, 100, 60)
    b2 = rand_rotated(g, 110, 100, 60)
    # structured cases: identical, same-centre different angle, axis-aligned neighbours, zero-area
    b2[:10] = b1[:10]
    b2[10:20, :4] = b1[10:20, :4]
    b1[20:30, 4] = 0
    b2[20:30, 4] = 90
    b1[30, 2] = 0.0
    b2[31] = torch.tensor([50.0, 50.0, 1e-8, 1e-8, 10.0])
    ious = D2.box_iou_rotated(b1, b2)
    dets = rand_rotated(g, 400, 120, 50)
    dets[100:180] = dets[:80] + torch.randn(80, 5, generator=g) * torch.tensor([2.0, 2.0, 2.0, 2.0, 5.0])
    dets[:, 2:4].clamp_(min=0.5)
    # no exact score ties here: the reference sorts with a non-stable `scores.sort(0, descending=True)`
    # (nms_rotated_cpu.cpp:26), so the order of tied scores is implementation-defined (probed: AVX sort
    # returns ties in reverse index order).  Tie behaviour is pinned separately as "stable, lower index first".
    scores = torch.rand(400, generator=g)
    idxs = torch.randint(0, 4, (400,), generator=g)
    out = {"b1": b1, "b2": b2, "ious": ious, "dets": dets, "scores": scores, "idxs": idxs,
           "thr": np.asarray([0.1, 0.3, 0.5, 0.7])}
    for i, t in enumerate([0.1, 0.3, 0.5, 0.7]):
        out[f"keep{i}"] = D2.nms_rotated(dets, scores, t)
    save("rotated", **out)


def gen_deform_conv():
    g = torch.Generator().manual_seed(2024)
    cases = [
        # n, cin, h, w, cout, k, stride, pad, dil, groups, dg, modulated, bias
        (2, 8, 10, 12, 8, 3, 1, 1, 1, 1, 1, False, False),
        (2, 8, 10, 12, 12, 3, 2, 1, 1, 2, 2, True, True),
        (1, 4, 9, 7, 6, 3, 1, 2, 2, 1, 1, True, False),
        (1, 6, 2, 2, 6, 3, 1, 1, 1, 3, 1, False, False),  # input smaller than kernel (test_deformable.py:112-133)
    ]
    out = {"cases": np.asarray([[int(v) for v in c] for c in cases])}
    for i, (n, cin, h, w, cout, k, s, p, d, grp, dg, mod, hb) in enumerate(cases):
        ho = (h + 2 * p - (d * (k - 1) + 1)) // s + 1
        wo = (w + 2 * p - (d * (k - 1) + 1)) // s + 1
        x = torch.randn(n, cin, h, w, generator=g, requires_grad=True)
        off = (torch.randn(n, 2 * dg * k * k, ho, wo, generator=g) * 1.5).requires_grad_(True)
        mask = torch.sigmoid(torch.randn(n, dg * k * k, ho, wo, generator=g)).requires_grad_(True) if mod else None
        wt = (torch.randn(cout, cin // grp, k, k, generator=g) * 0.2).requires_grad_(True)
        bias = torch.randn(cout, generator=g).requires_grad_(True) if hb else None
        y = torchvision.ops.deform_conv2d(x, off, wt, bias, stride=s, padding=p, dilation=d, mask=mask)
        go = torch.randn(y.shape, generator=g)
        y.backward(go)
        out.update({f"x{i}": x, f"off{i}": off, f"w{i}": wt, f"y{i}": y, f"go{i}": go,
                    f"gx{i}": x.grad, f"goff{i}": off.grad, f"gw{i}": wt.grad})
        if mod:
            out.update({f"mask{i}": mask, f"gmask{i}": mask.grad})
        if hb:
            out.update({f"bias{i}": bias, f"gbias{i}": bias.grad})
    save("deform_conv", **out)


def gen_paste_masks():
    spec = importlib.util.spec_from_file_location("ref_mask_ops", REF + "/detectron2/layers/mask_ops.py")
    mo = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mo)
    g = torch.Generator().manual_seed(42)
    n, m, h, w = 9, 28, 61, 83
    masks = torch.rand(n, m, m, generator=g)
    boxes = random_boxes(g, n, 60)
    boxes[0] = torch.tensor([-5.0, -7.5, 30.2, 20.1])  # partly outside
    boxes[1] = torch.tensor([10.0, 10.0, 10.0, 30.0])  # degenerate width (x1 == x0)
    boxes[2] = torch.tensor([70.0, 50.0, 120.0, 90.0])  # crosses the border
    boxes[3] = torch.tensor([20.3, 20.7, 21.1, 21.9])  # sub-pixel box
    out_bool = mo.paste_masks_in_image(masks, boxes, (h, w), threshold=0.5)
    out_u8 = mo.paste_masks_in_image(masks, boxes, (h, w), threshold=-1)
    soft, _ = mo._do_paste_mask(masks[:, None], boxes, h, w, skip_empty=False)
    save("paste_masks", masks=masks, boxes=boxes, hw=np.asarray([h, w]), out_bool=out_bool, out_u8=out_u8, soft=soft)


def _import_reference_proposal_utils():
    """The real detectron2 find_top_rpn_proposals, imported with stub fvcore / pycocotools (SURVEY Appendix B.3)."""
    import types

    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    sys.path.insert(0, REF)
    fv = stub("fvcore", __version__="0.1.5")
    fv.__path__ = []
    nn_ = stub("fvcore.nn")
    nn_.__path__ = []
    stub("fvcore.nn.distributed", differentiable_all_reduce=lambda x: x)
    nn_.weight_init = stub("fvcore.nn.weight_init", c2_msra_fill=lambda m: None, c2_xavier_fill=lambda m: None)
    pc = stub("pycocotools")
    pc.__path__ = []
    stub("pycocotools.mask")
    spec = importlib.util.spec_from_file_location(
        "ref_proposal_utils", REF + "/detectron2/modeling/proposal_generator/proposal_utils.py")
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def gen_rpn_proposals():
    ref = _import_reference_proposal_utils()
    g = torch.Generator().manual_seed(77)
    n, sizes = 2, [(120, 160), (100, 200)]
    per_level = [600, 300, 100]
    props, logits = [], []
    for a in per_level:
        ctr = torch.rand(n, a, 2, generator=g) * torch.tensor([220.0, 140.0]) - 10
        wh = torch.rand(n, a, 2, generator=g) * 60 + 0.5
        b = torch.cat([ctr - wh / 2, ctr + wh / 2], 2)
        props.append(b)
        logits.append(torch.randn(n, a, generator=g))
    props[0][0, 3] = float("nan")          # non-finite box
    logits[1][1, 5] = float("inf")         # non-finite score
    props[2][1, 7] = torch.tensor([50.0, 50.0, 50.5, 80.0])  # narrower than min_box_size
    logits[0][0, 10:14] = logits[0][0, 10]  # score ties
    out = {"sizes": np.asarray(sizes), "per_level": np.asarray(per_level), "cfg": np.asarray([0.7, 150, 60, 2.0])}
    for l in range(3):
        out[f"props{l}"] = props[l]
        out[f"logits{l}"] = logits[l]
    res = ref.find_top_rpn_proposals([p.clone() for p in props], [x.clone() for x in logits], sizes, 0.7, 150, 60, 2.0, False)
    for i, r in enumerate(res):
        out[f"boxes_img{i}"] = r.proposal_boxes.tensor
        out[f"scores_img{i}"] = r.objectness_logits
    save("rpn_proposals", **out)


def _import_reference_fast_rcnn():
    """The real detectron2 fast_rcnn_inference_single_image, imported with stubs for its unrelated dependencies."""
    import types

    _import_reference_proposal_utils()  # fvcore / pycocotools stubs + sys.path

    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    sys.modules["fvcore.nn"].giou_loss = sys.modules["fvcore.nn"].smooth_l1_loss = lambda *a, **k: None
    stub("detectron2.config", configurable=lambda f=None, **k: (f if f else (lambda g: g)))
    stub("detectron2.utils.events", get_event_storage=lambda: None)
    d = stub("detectron2.data")
    d.__path__ = []
    stub("detectron2.data.detection_utils", get_fed_loss_cls_weights=None)
    import detectron2.layers  # noqa: F401
    import detectron2.structures  # noqa: F401

    mm = stub("detectron2.modeling")
    mm.__path__ = []
    stub("detectron2.modeling.box_regression", Box2BoxTransform=object, _dense_box_regression_loss=None)
    spec = importlib.util.spec_from_file_location("ref_fast_rcnn", REF + "/detectron2/modeling/roi_heads/fast_rcnn.py")
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def gen_fast_rcnn_inference():
    ref = _import_reference_fast_rcnn()
    g = torch.Generator().manual_seed(31)
    out = {"cfg": np.asarray([0.05, 0.5, 25])}
    shapes = [(120, 160), (90, 200)]
    out["shapes"] = np.asarray(shapes)
    for i, (r, k, agnostic) in enumerate([(80, 6, False), (50, 6, True)]):
        base = torch.rand(12, 4, generator=g) * torch.tensor([150.0, 100.0, 60.0, 50.0])
        base[:, 2:] += base[:, :2] + 5
        pick = torch.randint(0, 12, (r,), generator=g)
        nb = 1 if agnostic else k
        boxes = (base[pick][:, None, :] + torch.randn(r, nb, 4, generator=g) * 4).reshape(r, nb * 4)
        scores = torch.softmax(torch.randn(r, k + 1, generator=g) * 2.5, dim=1)
        if i == 0:
            boxes[7, 2] = float("inf")       # invalid row (dropped before everything else)
            scores[9] = float("nan")
            scores[20, 1] = scores[21, 1]    # tie
        res, rows = ref.fast_rcnn_inference_single_image(boxes.clone(), scores.clone(), shapes[i], 0.05, 0.5, 25)
        out.update({f"boxes{i}": boxes, f"scores{i}": scores, f"out_boxes{i}": res.pred_boxes.tensor,
                    f"out_scores{i}": res.scores, f"out_classes{i}": res.pred_classes, f"out_rows{i}": rows})
    save("fast_rcnn_inference", **out)


def _import_reference_dense_detector():
    """The real DenseDetector decode methods + Box2BoxTransform, imported with stubs for their unrelated dependencies."""
    import types

    _import_reference_fast_rcnn()  # fvcore / pycocotools / config / events / data stubs, detectron2.layers + structures

    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    sys.modules["detectron2.data.detection_utils"].convert_image_to_rgb = None
    mm = sys.modules["detectron2.modeling"]
    mm.Backbone = object
    spec = importlib.util.spec_from_file_location("detectron2.modeling.box_regression",
                                                  REF + "/detectron2/modeling/box_regression.py")
    br = importlib.util.module_from_spec(spec)
    sys.modules["detectron2.modeling.box_regression"] = br
    spec.loader.exec_module(br)
    ma = stub("detectron2.modeling.meta_arch")
    ma.__path__ = []
    stub("detectron2.modeling.postprocessing", detector_postprocess=None)
    spec = importlib.util.spec_from_file_location("detectron2.modeling.meta_arch.dense_detector",
                                                  REF + "/detectron2/modeling/meta_arch/dense_detector.py")
    dd = importlib.util.module_from_spec(spec)
    sys.modules["detectron2.modeling.meta_arch.dense_detector"] = dd
    spec.loader.exec_module(dd)
    return dd, br


def gen_retinanet_inference():
    """RetinaNet.forward_inference (meta_arch/retinanet.py:256-308) on the real DenseDetector decode methods."""
    import types

    dd, br = _import_reference_dense_detector()  # also puts the reference checkout on sys.path
    from detectron2.layers import batched_nms
    from detectron2.structures import Boxes

    g = torch.Generator().manual_seed(2024)
    n, k_cls = 2, 5
    image_sizes = [(96, 128), (80, 120)]
    per_level = [(12 * 16 * 3, 8.0), (6 * 8 * 3, 16.0), (3 * 4 * 3, 32.0)]  # (H*W*A anchors, stride)
    score_thresh, topk_candidates, nms_thresh, max_det = 0.3, 60, 0.5, 20
    anchors, logits, deltas = [], [], []
    for r, stride in per_level:
        ctr = torch.rand(r, 2, generator=g) * torch.tensor([128.0, 96.0])
        wh = stride * (2 + 4 * torch.rand(r, 2, generator=g))
        anchors.append(torch.cat([ctr - wh / 2, ctr + wh / 2], 1))
        logits.append(torch.randn(n, r, k_cls, generator=g) * 1.5 - 1.0)
        deltas.append(torch.randn(n, r, 4, generator=g) * 0.3)
    deltas[0][0, 5, 2] = 9.0      # exercises the scale clamp (box_regression.py:103)
    logits[2][1] = -20.0          # a level without any candidate for image 1
    me = types.SimpleNamespace(box2box_transform=br.Box2BoxTransform(weights=(1.0, 1.0, 1.0, 1.0)))
    me._decode_per_level_predictions = types.MethodType(dd.DenseDetector._decode_per_level_predictions, me)
    out = {"cfg": np.asarray([score_thresh, topk_candidates, nms_thresh, max_det]), "image_sizes": np.asarray(image_sizes)}
    for l in range(len(per_level)):
        out[f"anchors{l}"], out[f"logits{l}"], out[f"deltas{l}"] = anchors[l], logits[l], deltas[l]
    for img_idx, image_size in enumerate(image_sizes):
        scores_per_image = [x[img_idx].clone().sigmoid_() for x in logits]      # retinanet.py:267
        deltas_per_image = [x[img_idx] for x in deltas]
        pred = dd.DenseDetector._decode_multi_level_predictions(
            me, [Boxes(a) for a in anchors], scores_per_image, deltas_per_image, score_thresh, topk_candidates, image_size)
        keep = batched_nms(pred.pred_boxes.tensor, pred.scores, pred.pred_classes, nms_thresh)  # retinanet.py:305-307
        res = pred[keep[:max_det]]                                                              # :308
        out[f"n_candidates{img_idx}"] = np.asarray(len(pred))
        out[f"out_boxes{img_idx}"] = res.pred_boxes.tensor
        out[f"out_scores{img_idx}"] = res.scores
        out[f"out_classes{img_idx}"] = res.pred_classes
    save("retinanet_inference", **out)


def gen_postprocessing():
    """detector_postprocess (modeling/postprocessing.py:9-74) and BitMasks.crop_and_resize (structures/masks.py:193-224),
    both from the real reference modules (CPU: torchvision roi_align, python paste)."""
    _import_reference_fast_rcnn()  # stubs + sys.path
    from detectron2.structures import BitMasks, Boxes, Instances

    spec = importlib.util.spec_from_file_location("ref_postprocessing", REF + "/detectron2/modeling/postprocessing.py")
    pp = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(pp)
    g = torch.Generator().manual_seed(808)
    n, m, h, w, oh, ow = 11, 28, 60, 90, 97, 141
    boxes = random_boxes(g, n, 60)
    boxes[:, 0::2] *= 1.4
    boxes[0] = torch.tensor([10.0, 10.0, 10.0, 30.0])       # empty after scaling (zero width)
    boxes[1] = torch.tensor([85.0, 50.0, 120.0, 70.0])      # clipped by the image border
    boxes[2] = torch.tensor([95.0, 5.0, 130.0, 20.0])       # entirely outside -> empty after clipping
    scores, classes = torch.rand(n, generator=g), torch.randint(0, 7, (n,), generator=g)
    masks = torch.rand(n, 1, m, m, generator=g)
    inst = Instances((h, w), pred_boxes=Boxes(boxes.clone()), scores=scores.clone(), pred_classes=classes.clone(),
                     pred_masks=masks.clone())
    res = pp.detector_postprocess(inst, oh, ow, 0.5)
    out = {"hw": np.asarray([h, w, oh, ow]), "boxes": boxes, "scores": scores, "classes": classes, "masks": masks,
           "out_boxes": res.pred_boxes.tensor, "out_scores": res.scores, "out_classes": res.pred_classes,
           "out_masks": res.pred_masks}
    # crop_and_resize: ground-truth bitmasks (filled ellipses) cropped by jittered boxes
    k, gh, gw, ms = 9, 72, 104, 28
    yy, xx = torch.meshgrid(torch.arange(gh, dtype=torch.float32), torch.arange(gw, dtype=torch.float32), indexing="ij")
    cb = random_boxes(g, k, 70)
    cb[:, 0::2] *= 1.4
    bit = torch.zeros(k, gh, gw, dtype=torch.bool)
    for i in range(k):
        cx, cy = (cb[i, 0] + cb[i, 2]) / 2, (cb[i, 1] + cb[i, 3]) / 2
        rx, ry = (cb[i, 2] - cb[i, 0]) / 2 + 0.5, (cb[i, 3] - cb[i, 1]) / 2 + 0.5
        bit[i] = ((xx - cx) / rx) ** 2 + ((yy - cy) / ry) ** 2 <= 1.0
    crop_boxes = cb + torch.randn(k, 4, generator=g) * 2
    out.update({"bit_masks": bit, "crop_boxes": crop_boxes,
                "crops": BitMasks(bit).crop_and_resize(crop_boxes, ms), "mask_size": np.asarray(ms)})
    save("postprocessing", **out)


def gen_compiled_reference():
    """box_iou_rotated / nms_rotated and roi_align_rotated forward + backward of the compiled reference csrc, at the inputs of
    the cross-checks in tests/test_oracle_pins.py (test_live_vs_compiled_reference, test_sweep_roi_align_rotated_*)."""
    g = torch.Generator().manual_seed(11)
    n = 150
    b = torch.stack([torch.rand(n, generator=g) * 80, torch.rand(n, generator=g) * 80, 1 + torch.rand(n, generator=g) * 40,
                     1 + torch.rand(n, generator=g) * 40, (torch.rand(n, generator=g) - 0.5) * 400], 1)
    out = {"b": b, "ious": D2.box_iou_rotated(b, b.flip(0))}
    out["s"] = s = torch.rand(n, generator=g)
    out["thr"] = thrs = np.asarray([0.2, 0.5])
    for i, thr in enumerate(thrs):
        out[f"keep{i}"] = D2.nms_rotated(b, s, float(thr))
    for seed in range(3):
        g = torch.Generator().manual_seed(3000 + seed)
        n, c, h, w = 2, 3 + seed, 17 + 5 * seed, 23
        ph, pw, sr = [(7, 7, 0), (3, 5, 2), (2, 2, 3)][seed]
        k = 19
        rois = torch.cat([torch.randint(0, n, (k, 1), generator=g).float(),
                          torch.rand(k, 2, generator=g) * torch.tensor([w * 4.0, h * 4.0]),
                          2 + torch.rand(k, 2, generator=g) * 50, (torch.rand(k, 1, generator=g) - 0.5) * 360], 1)
        x = torch.randn(n, c, h, w, generator=g)
        y = D2.roi_align_rotated_forward(x, rois, 0.25, ph, pw, sr)
        go = torch.randn(y.shape, generator=g)
        out.update({f"sweep{seed}_cfg": np.asarray([ph, pw, sr]), f"sweep{seed}_x": x, f"sweep{seed}_rois": rois,
                    f"sweep{seed}_y": y, f"sweep{seed}_go": go,
                    f"sweep{seed}_gx": D2.roi_align_rotated_backward(go, rois, 0.25, ph, pw, n, c, h, w, sr)})
    save("compiled_reference", **out)


def gen_paste_masks_random():
    """The reference's paste_masks_in_image on random masks and boxes inside a 150 x 200 image (the cross-check of
    oracle/paste_ref.py in tests/test_oracle_pins.py)."""
    spec = importlib.util.spec_from_file_location("ref_mask_ops", REF + "/detectron2/layers/mask_ops.py")
    mo = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mo)
    g = torch.Generator().manual_seed(8)
    masks = torch.rand(6, 28, 28, generator=g)
    ctr = torch.rand(6, 2, generator=g) * torch.tensor([200.0, 150.0])
    wh = 10 + torch.rand(6, 2, generator=g) * 90
    boxes = torch.cat([ctr - wh / 2, ctr + wh / 2], 1)
    save("paste_masks_random", masks=masks, boxes=boxes, hw=np.asarray([150, 200]),
         out_bool=mo.paste_masks_in_image(masks, boxes, (150, 200), 0.5))


def gen_reference_shim_protocol():
    """The calls that the reference's deform-conv autograd Functions (detectron2/layers/deform_conv.py, `_DeformConv` and
    `_ModulatedDeformConv`) make into `detectron2._C`, recorded through a stand-in module: which input goes into which
    argument, the shape of every buffer the caller allocates and whether it is zero when passed, every scalar argument, and
    which buffer each Function returns as its output or as each gradient.  tests/test_reference_shim.py replays the record
    against the signatures of detectron2_b200._C."""
    import json
    import math
    import types

    class FakeCuda(torch.Tensor):  # the reference Functions refuse CPU tensors; they only test the flag
        @property
        def is_cuda(self):
            return True

    def fc(t):
        return torch.Tensor._make_subclass(FakeCuda, t, t.requires_grad)

    def plain(t):
        return t.detach().as_subclass(torch.Tensor)

    g = torch.Generator().manual_seed(0)
    n, c, h, w, co = 2, 4, 7, 9, 6
    inputs = {"x": torch.randn(n, c, h, w, generator=g), "off": torch.randn(n, 18, h, w, generator=g),
              "mask": torch.sigmoid(torch.randn(n, 9, h, w, generator=g)),
              "w": torch.randn(co, c, 3, 3, generator=g) * (1 / math.sqrt(c * 9)), "bias": torch.randn(co, generator=g),
              "go": torch.randn(n, co, h, w, generator=g)}
    calls, buffers = [], {}  # buffers: id(tensor) -> (buffer number, tensor kept alive so that ids stay unique)

    def encode(a):
        if not isinstance(a, torch.Tensor):
            assert a is None or isinstance(a, (bool, int, float)), type(a)
            return a
        p = plain(a)
        for name, t in inputs.items():
            if p.shape == t.shape and torch.equal(p, t):
                return {"input": name}
        if id(a) not in buffers:
            buffers[id(a)] = (len(buffers), a)
        return {"buffer": buffers[id(a)][0], "shape": list(p.shape), "zero": bool((p == 0).all())}

    def recorder(name):
        def fn(*args, **kwargs):
            assert not kwargs, (name, kwargs)
            calls.append({"fn": name, "args": [encode(a) for a in args]})
            for a in args:  # every buffer a call writes holds its buffer number + 1 afterwards: identifies what is returned
                if isinstance(a, torch.Tensor) and id(a) in buffers and a.numel():
                    with torch.no_grad():
                        a.fill_(buffers[id(a)][0] + 1)
            return 1
        return fn

    shim = types.ModuleType("detectron2._C")
    for name in ("deform_conv_forward", "deform_conv_backward_input", "deform_conv_backward_filter",
                 "modulated_deform_conv_forward", "modulated_deform_conv_backward"):
        setattr(shim, name, recorder(name))
    shim.get_cuda_version, shim.has_cuda, shim.get_compiler_version = (lambda: "CUDA"), (lambda: True), (lambda: "nvcc")

    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    for k in [k for k in sys.modules if k.startswith(("detectron2", "fvcore"))]:
        del sys.modules[k]
    fv = stub("fvcore", __version__="0.1.5")
    fv.nn = stub("fvcore.nn")
    stub("fvcore.nn.distributed", differentiable_all_reduce=lambda x: x)
    fv.nn.weight_init = stub("fvcore.nn.weight_init")
    sys.path.insert(0, REF)
    import detectron2  # noqa: F401  (the real package __init__)

    sys.modules["detectron2._C"] = shim
    detectron2._C = shim
    mod = importlib.import_module("detectron2.layers.deform_conv")

    def returned(t):
        v = plain(t).unique()
        assert v.numel() == 1, "returned tensor is not one recorded buffer"
        return int(v.item()) - 1

    x, off, mask, wt, bias, go = (inputs[k] for k in ("x", "off", "mask", "w", "bias", "go"))
    roles = {}
    xs = [fc(t.clone().requires_grad_(True)) for t in (x, off, wt)]
    y = mod.deform_conv(xs[0], xs[1], xs[2], 1, 1, 1, 1, 1, 64)
    y.backward(fc(go))
    roles["v1"] = dict(zip(("y", "x", "off", "w"), [returned(t) for t in [y] + [a.grad for a in xs]]))
    xs = [fc(t.clone().requires_grad_(True)) for t in (x, off, mask, wt, bias)]
    y = mod.modulated_deform_conv(xs[0], xs[1], xs[2], xs[3], xs[4], 1, 1, 1, 1, 1)
    y.backward(fc(go))
    roles["v2"] = dict(zip(("y", "x", "off", "mask", "w", "bias"), [returned(t) for t in [y] + [a.grad for a in xs]]))
    save("reference_shim_protocol", protocol=np.asarray(json.dumps({"calls": calls, "returns": roles})), **inputs)


GENERATORS = {"roi_align": gen_roi_align, "roi_align_rotated": gen_roi_align_rotated, "nms": gen_nms,
              "rotated": gen_rotated_iou_nms, "deform_conv": gen_deform_conv, "paste_masks": gen_paste_masks,
              "rpn_proposals": gen_rpn_proposals, "fast_rcnn_inference": gen_fast_rcnn_inference,
              "retinanet_inference": gen_retinanet_inference, "postprocessing": gen_postprocessing,
              "compiled_reference": gen_compiled_reference, "paste_masks_random": gen_paste_masks_random,
              "reference_shim_protocol": gen_reference_shim_protocol}

if __name__ == "__main__":
    torch.set_num_threads(1)
    for name in sys.argv[1:] or list(GENERATORS):
        GENERATORS[name]()
