"""Pins the CPU oracle (oracle/d2_oracle.c) to the reference BEFORE it is trusted as the checker.

Three layers of evidence (all CPU, `-m "not gpu"`):
  1. the reference's own known-answer tables (cited per test),
  2. the committed golden fixtures generated from torchvision CPU / the compiled reference CPU csrc /
     the reference python paste_masks (tests/golden/make_golden.py),
  3. cross-checks against torchvision CPU (live) and the compiled reference CPU csrc (results stored by make_golden.py).
"""
import math

import numpy as np
import pytest
import torch

from oracle import oracle as orc

T = torch.from_numpy


# ---------------------------------------------------------------- 1. reference known-answer tables
def _simple(img, box, res, aligned=True, sr=0):
    x = torch.as_tensor(img, dtype=torch.float32)[None, None]
    rois = torch.tensor([[0.0] + list(box)], dtype=torch.float32)
    return orc.roi_align_forward(x, rois, 1.0, res[0], res[1], sr, aligned)[0, 0]


def test_kat_roi_align_tables():  # /root/reference/tests/layers/test_roi_align.py:14-47
    img = np.arange(25).reshape(5, 5).astype("float32")
    old = [[7.5, 8, 8.5, 9], [10, 10.5, 11, 11.5], [12.5, 13, 13.5, 14], [15, 15.5, 16, 16.5]]
    new = [[4.5, 5.0, 5.5, 6.0], [7.0, 7.5, 8.0, 8.5], [9.5, 10.0, 10.5, 11.0], [12.0, 12.5, 13.0, 13.5]]
    assert np.allclose(_simple(img, [1, 1, 3, 3], (4, 4), aligned=False).numpy(), old)
    assert np.allclose(_simple(img, [1, 1, 3, 3], (4, 4), aligned=True).numpy(), new)


def test_kat_roi_align_empty_box():  # test_roi_align.py:111-121
    img = np.random.RandomState(0).rand(5, 5)
    o = _simple(img, [3, 4, 5, 4], (7, 7))
    assert o.shape == (7, 7) and (o == 0).all()
    rois = torch.tensor([[0.0, 3, 4, 5, 4]])
    gx = orc.roi_align_backward(torch.ones(1, 1, 7, 7), rois, 1.0, 7, 7, 1, 1, 5, 5, 0, True)
    assert (gx == 0).all()


def test_kat_roi_align_rotated_tables():  # test_roi_align_rotated.py:30-71
    img = torch.arange(25, dtype=torch.float32).reshape(5, 5)
    exp = torch.tensor([[4.5, 5.0, 5.5, 6.0], [7.0, 7.5, 8.0, 8.5], [9.5, 10.0, 10.5, 11.0], [12.0, 12.5, 13.0, 13.5]])

    def rot90(t, num):
        for _ in range(num % 4):
            t = t.transpose(0, 1).flip(0)
        return t

    for i in range(4):
        rois = torch.tensor([[0, 2.0, 2.0, 2.0, 2.0, 90.0 * i]])
        out = orc.roi_align_rotated_forward(img[None, None], rois, 1.0, 4, 4, 0)[0, 0]
        assert torch.allclose(out, rot90(exp, -i), atol=1e-5)
    out = orc.roi_align_rotated_forward(torch.rand(1, 1, 5, 5), torch.tensor([[0, 2.0, 3, 0, 0, 0]]), 1.0, 7, 7, 0)
    assert (out == 0).all()  # :102-105


def test_kat_deform_conv_tables():  # /root/reference/tests/layers/test_deformable.py:16-58
    x = torch.arange(25, dtype=torch.float32).reshape(1, 1, 5, 5)
    off = torch.full((1, 18, 5, 5), 0.5)
    w = torch.ones(1, 1, 3, 3)
    exp = np.array([[30, 41.25, 48.75, 45, 28.75], [62.25, 81, 90, 80.25, 50.25], [99.75, 126, 135, 117.75, 72.75],
                    [105, 131.25, 138.75, 120, 73.75], [71.75, 89.25, 93.75, 80.75, 49.5]])
    y = orc.deform_conv_forward(x, off, None, w, None, 1, 1, 1, 1, 1)
    assert np.allclose(y.numpy().reshape(5, 5), exp)
    y2 = orc.deform_conv_forward(x, off, torch.full((1, 9, 5, 5), 0.5), w, None, 1, 1, 1, 1, 1)
    assert np.allclose(y2.numpy().reshape(5, 5), exp * 0.5)


IOU_KATS = [  # /root/reference/tests/structures/test_rotated_boxes.py
    ([[0.5, 0.5, 1.0, 1.0, 0.0]], [[0.25, 0.5, 0.5, 1.0, 0.0]], [[0.5]]),  # :46-51
    ([[565, 565, 10, 10.0, 0]], [[565, 565, 10, 8.3, 0]], [[0.83]]),  # :62-69
    ([[296.6620178222656, 458.73883056640625, 23.515729904174805, 47.677001953125, 0.08795166015625]],
     [[296.66201, 458.73882000000003, 23.51573, 47.67702, 0.087951]], [[1.0]]),  # :97-117 (#2154)
    ([[2563.74462890625, 1436.7901611328125, 2174.703369140625, 214.09500122070312, 115.11834716796875]],
     [[2563.74462890625, 1436.790283203125, 2174.702880859375, 214.09495544433594, 115.11835479736328]],
     [[1.0]]),  # :119-147 (#2167)
    ([[1, 1, math.sqrt(2), math.sqrt(2), 45], [1, 1, 2 * math.sqrt(2), 2 * math.sqrt(2), -45]], [[1, 1, 2, 2, 0]],
     [[0.5], [0.5]]),  # :276-290
    ([[5, 5, 10, 6, 55]], [[5, 5, 10, 6, -35]], [[36.0 / (36 + 24 + 24)]]),  # :292-299
    ([[299.5, 417.370422, 600.0, 364.259186, 27.1828]], [[299.5, 417.370422, 600.0, 364.259155, 27.1828]],
     [[364.259155 / 364.259186]]),  # :301-317
    ([[3, 3, 8, 2, -45.0]], [[6, 0, 8, 2, -45.0]], [[0.0]]),  # :347-357 (#1207 simplified)
    ([[160.0, 153.0, 230.0, 23.0, -37.0]], [[190.0, 127.0, 80.0, 21.0, -46.0]], [[0.0]]),  # :359-369 (#1207)
]


@pytest.mark.parametrize("b1,b2,exp", IOU_KATS)
def test_kat_rotated_iou(b1, b2, exp):
    out = orc.box_iou_rotated(torch.tensor(b1, dtype=torch.float32), torch.tensor(b2, dtype=torch.float32))
    assert torch.allclose(out, torch.tensor(exp, dtype=torch.float32))


def test_kat_rotated_iou_0deg_and_many():  # :247-274, :319-345
    b1 = torch.tensor([[0.5, 0.5, 1.0, 1.0, 0.0]] * 2)
    b2 = torch.tensor([[0.5, 0.5, 1.0, 1.0, 0.0], [0.25, 0.5, 0.5, 1.0, 0.0], [0.5, 0.25, 1.0, 0.5, 0.0],
                       [0.25, 0.25, 0.5, 0.5, 0.0], [0.75, 0.75, 0.5, 0.5, 0.0], [1.0, 1.0, 1.0, 1.0, 0.0]])
    exp = torch.tensor([[1.0, 0.5, 0.5, 0.25, 0.25, 0.25 / (2 - 0.25)]] * 2)
    assert torch.allclose(orc.box_iou_rotated(b1, b2), exp)
    n1, n2 = 100, 200
    bb1 = torch.tensor([[5 + 20 * i, 5 + 20 * i, 10, 10, 0] for i in range(n1)], dtype=torch.float32)
    bb2 = torch.tensor([[5 + 20 * i, 5 + 20 * i, 10, 1 + 9 * i / n2, 0] for i in range(n2)], dtype=torch.float32)
    exp = torch.zeros(n1, n2)
    for i in range(n1):
        exp[i, i] = (1 + 9 * i / n2) / 10.0
    assert torch.allclose(orc.box_iou_rotated(bb1, bb2), exp)


def test_kat_rotated_iou_extreme_nonnegative():  # :80-95 (#1266)
    b1 = torch.tensor([[160.0, 153.0, 230.0, 23.0, -37.0]])
    b2 = torch.tensor([[-1.117407639806935e17, 1.3858420478349148e18, 1000.0000610351562, 1000.0000610351562, 1612.0]])
    assert orc.box_iou_rotated(b1, b2).min() >= 0


def test_kat_nms_rotated_vs_horizontal():  # /root/reference/tests/layers/test_nms_rotated.py:73-116 semantics
    g = torch.Generator().manual_seed(0)
    n = 300
    boxes = torch.rand(n, 4, generator=g) * 100
    boxes[:, 2:] += boxes[:, :2] + 1
    scores = torch.rand(n, generator=g)
    rot = torch.zeros(n, 5)
    rot[:, 0] = (boxes[:, 0] + boxes[:, 2]) / 2
    rot[:, 1] = (boxes[:, 1] + boxes[:, 3]) / 2
    rot[:, 2] = boxes[:, 2] - boxes[:, 0]
    rot[:, 3] = boxes[:, 3] - boxes[:, 1]
    for thr in [0.2, 0.5, 0.8]:
        kh = orc.nms(boxes, scores, thr).tolist()
        kr = orc.nms_rotated(rot, scores, thr).tolist()
        # the reference allows an edit distance <= 1 here; identical sets expected in practice
        assert len(set(kh) ^ set(kr)) <= 1


# ---------------------------------------------------------------- 2. committed fixtures
def test_golden_roi_align(golden):
    d = golden("roi_align")
    x, rois = T(d["x"]), T(d["rois"])
    for i, (ph, pw, sr, al) in enumerate(d["cfgs"]):
        y = orc.roi_align_forward(x, rois, 0.5, int(ph), int(pw), int(sr), bool(al))
        assert torch.allclose(y, T(d[f"y{i}"]), rtol=1e-4, atol=1e-5), i
        gx = orc.roi_align_backward(T(d[f"go{i}"]), rois, 0.5, int(ph), int(pw), 2, 8, 24, 32, int(sr), bool(al))
        assert torch.allclose(gx, T(d[f"gx{i}"]), rtol=1e-4, atol=1e-4), i


def test_golden_roi_align_rotated(golden):
    d = golden("roi_align_rotated")
    x, rois = T(d["x"]), T(d["rois"])
    for i, (ph, pw, sr) in enumerate(d["cfgs"]):
        y = orc.roi_align_rotated_forward(x, rois, 0.5, int(ph), int(pw), int(sr))
        assert torch.allclose(y, T(d[f"y{i}"]), rtol=1e-4, atol=1e-5), i
        gx = orc.roi_align_rotated_backward(T(d[f"go{i}"]), rois, 0.5, int(ph), int(pw), 2, 6, 20, 28, int(sr))
        assert torch.allclose(gx, T(d[f"gx{i}"]), rtol=1e-4, atol=1e-4), i


def test_golden_nms_bit_exact(golden):
    d = golden("nms")
    boxes, scores, idxs = T(d["boxes"]), T(d["scores"]), T(d["idxs"])
    for i, t in enumerate(d["thr"]):
        assert torch.equal(orc.nms(boxes, scores, float(t)), T(d[f"keep{i}"]))
        assert torch.equal(orc.batched_nms(boxes, scores, idxs, float(t)), T(d[f"bkeep_trick{i}"]))


def test_golden_rotated_bit_exact(golden):
    d = golden("rotated")
    ious = orc.box_iou_rotated(T(d["b1"]), T(d["b2"]))
    assert np.array_equal(ious.numpy().view(np.uint32), d["ious"].view(np.uint32))  # bit-exact
    for i, t in enumerate(d["thr"]):
        assert torch.equal(orc.nms_rotated(T(d["dets"]), T(d["scores"]), float(t)), T(d[f"keep{i}"]))


def test_golden_deform_conv(golden):
    d = golden("deform_conv")
    for i, (n, cin, h, w, cout, k, s, p, dil, grp, dg, mod, hb) in enumerate(d["cases"]):
        x, off, wt = T(d[f"x{i}"]), T(d[f"off{i}"]), T(d[f"w{i}"])
        mask = T(d[f"mask{i}"]) if mod else None
        bias = T(d[f"bias{i}"]) if hb else None
        y = orc.deform_conv_forward(x, off, mask, wt, bias, int(s), int(p), int(dil), int(grp), int(dg))
        assert torch.allclose(y, T(d[f"y{i}"]), rtol=1e-4, atol=1e-4), i
        gx, goff, gmask, gw, gb = orc.deform_conv_backward(x, off, mask, wt, T(d[f"go{i}"]), int(s), int(p), int(dil),
                                                           int(grp), int(dg), bool(hb))
        assert torch.allclose(gx, T(d[f"gx{i}"]), rtol=1e-4, atol=1e-4), i
        assert torch.allclose(goff, T(d[f"goff{i}"]), rtol=1e-4, atol=1e-4), i
        assert torch.allclose(gw, T(d[f"gw{i}"]), rtol=1e-4, atol=1e-4), i
        if mod:
            assert torch.allclose(gmask, T(d[f"gmask{i}"]), rtol=1e-4, atol=1e-4), i
        if hb:
            assert torch.allclose(gb, T(d[f"gbias{i}"]), rtol=1e-4, atol=1e-4), i


def test_golden_paste_masks(golden):
    d = golden("paste_masks")
    h, w = [int(v) for v in d["hw"]]
    ob, soft = orc.paste_masks(T(d["masks"]), T(d["boxes"]), (h, w), 0.5, return_soft=True)
    ref_soft = T(d["soft"])
    finite = torch.isfinite(ref_soft)
    assert torch.allclose(soft[finite], ref_soft[finite], rtol=1e-5, atol=1e-6)
    # boolean output must agree everywhere except where the soft value sits on the threshold
    mism = ob != T(d["out_bool"])
    assert not (mism & ((ref_soft - 0.5).abs() > 1e-5)).any()
    assert mism.sum() <= 2
    ou = orc.paste_masks(T(d["masks"]), T(d["boxes"]), (h, w), -1.0)
    diff = (ou.int() - T(d["out_u8"]).int()).abs()
    assert diff.max() <= 1 and (diff > 0).float().mean() < 1e-3


# ---------------------------------------------------------------- 3. live cross-checks
def test_live_vs_torchvision():
    tv = pytest.importorskip("torchvision")
    g = torch.Generator().manual_seed(5)
    x = torch.randn(1, 16, 50, 76, generator=g)
    k = 64
    cx, cy = torch.rand(k, generator=g) * 304, torch.rand(k, generator=g) * 200
    w, h = 4 + torch.rand(k, generator=g) * 150, 4 + torch.rand(k, generator=g) * 150
    rois = torch.stack([torch.zeros(k), cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1)
    for sr in (0, 2):
        ref = tv.ops.roi_align(x, rois, (7, 7), 0.25, sr, True)
        assert torch.allclose(orc.roi_align_forward(x, rois, 0.25, 7, 7, sr, True), ref, rtol=1e-4, atol=1e-5)
    boxes = torch.rand(2000, 4, generator=g) * 400
    boxes[:, 2:] = boxes[:, :2] + torch.rand(2000, 2, generator=g) * 120 + 1
    scores = torch.rand(2000, generator=g)
    for thr in (0.3, 0.5, 0.7):
        assert torch.equal(orc.nms(boxes, scores, thr), tv.ops.nms(boxes, scores, thr))


def test_live_vs_compiled_reference(golden):
    """box_iou_rotated / nms_rotated against what the compiled reference csrc returned (fixture from make_golden.py)."""
    d = golden("compiled_reference")
    b, s = T(d["b"]), T(d["s"])
    got = orc.box_iou_rotated(b, b.flip(0))
    assert np.array_equal(got.numpy().view(np.uint32), d["ious"].view(np.uint32))
    for i, thr in enumerate(d["thr"]):
        assert torch.equal(orc.nms_rotated(b, s, float(thr)), T(d[f"keep{i}"]))


def test_paste_port_matches_fixture_and_reference(golden):
    """oracle/paste_ref.py (the CPU-baseline port) against the golden fixture, and against what the real reference
    function returned on random masks and boxes (fixture from make_golden.py)."""
    from oracle import paste_ref

    d = golden("paste_masks")
    h, w = [int(v) for v in d["hw"]]
    got = paste_ref.paste_masks_in_image_cpu(T(d["masks"]), T(d["boxes"]), (h, w), 0.5)
    keep = [i for i in range(9) if i != 1]  # box 1 is degenerate (x1 == x0): nan grid, not a baseline case
    assert torch.equal(got[keep], T(d["out_bool"])[keep])
    d = golden("paste_masks_random")
    h, w = [int(v) for v in d["hw"]]
    assert torch.equal(paste_ref.paste_masks_in_image_cpu(T(d["masks"]), T(d["boxes"]), (h, w), 0.5), T(d["out_bool"]))


def _rpn_fixture(golden):
    d = golden("rpn_proposals")
    props = [T(d[f"props{l}"]) for l in range(3)]
    logits = [T(d[f"logits{l}"]) for l in range(3)]
    sizes = [tuple(int(v) for v in r) for r in d["sizes"]]
    thr, pre, post, mbs = d["cfg"]
    return d, props, logits, sizes, float(thr), int(pre), int(post), float(mbs)


def test_golden_rpn_proposals(golden):
    """oracle/proposals_ref.py against the REAL detectron2 find_top_rpn_proposals (fixture from make_golden.py)."""
    from oracle import proposals_ref

    d, props, logits, sizes, thr, pre, post, mbs = _rpn_fixture(golden)
    res = proposals_ref.find_top_rpn_proposals(props, logits, sizes, thr, pre, post, mbs, False)
    for i, (b, s) in enumerate(res):
        assert torch.equal(b, T(d[f"boxes_img{i}"])) and torch.equal(s, T(d[f"scores_img{i}"])), i


# ---------------------------------------------------------------- 4. randomized sweeps (oracle vs torchvision / compiled reference)
@pytest.mark.parametrize("seed", range(6))
def test_sweep_roi_align_fwd_bwd_vs_torchvision(seed):
    tv = pytest.importorskip("torchvision")
    g = torch.Generator().manual_seed(1000 + seed)
    n, c = int(torch.randint(1, 4, (1,), generator=g)), int(torch.randint(1, 9, (1,), generator=g))
    h, w = int(torch.randint(5, 40, (1,), generator=g)), int(torch.randint(5, 40, (1,), generator=g))
    ph, pw = int(torch.randint(1, 9, (1,), generator=g)), int(torch.randint(1, 9, (1,), generator=g))
    sr, aligned = int(torch.randint(0, 4, (1,), generator=g)), bool(seed % 2)
    scale = [1.0, 0.5, 0.25][seed % 3]
    k = 23
    ctr = torch.rand(k, 2, generator=g) * torch.tensor([w / scale, h / scale])
    wh = torch.rand(k, 2, generator=g) * torch.tensor([w / scale, h / scale]) * 0.8
    rois = torch.cat([torch.randint(0, n, (k, 1), generator=g).float(), ctr - wh / 2, ctr + wh / 2], 1)
    rois[0, 1:] = torch.tensor([-30.0, -20.0, 2 * w / scale, 2 * h / scale])  # far larger than the map
    x = torch.randn(n, c, h, w, generator=g).requires_grad_(True)
    ref = tv.ops.roi_align(x, rois, (ph, pw), scale, sr, aligned)
    got = orc.roi_align_forward(x.detach(), rois, scale, ph, pw, sr, aligned)
    assert torch.allclose(got, ref.detach(), rtol=1e-4, atol=1e-5), (got - ref.detach()).abs().max()
    go = torch.randn(ref.shape, generator=g)
    ref.backward(go)
    gx = orc.roi_align_backward(go, rois, scale, ph, pw, n, c, h, w, sr, aligned)
    assert torch.allclose(gx, x.grad, rtol=1e-4, atol=1e-4), (gx - x.grad).abs().max()


@pytest.mark.parametrize("seed", range(4))
def test_sweep_batched_nms_vs_torchvision(seed):
    tv = pytest.importorskip("torchvision")
    g = torch.Generator().manual_seed(2000 + seed)
    m, ncls = [17, 300, 999, 64][seed], [1, 3, 20, 64][seed]
    base = torch.rand(max(m // 6, 1), 4, generator=g) * 200
    base[:, 2:] = base[:, :2] + 5 + torch.rand(base.shape[0], 2, generator=g) * 80
    boxes = base[torch.randint(0, base.shape[0], (m,), generator=g)] + torch.randn(m, 4, generator=g) * 3
    boxes[:, 2:] = torch.maximum(boxes[:, 2:], boxes[:, :2] + 1)
    boxes.clamp_(min=0)  # detectron2 call sites clip first (see DESIGN 2, batched NMS note)
    scores = torch.rand(m, generator=g)
    idxs = torch.randint(0, ncls, (m,), generator=g)
    for thr in (0.3, 0.6):
        assert torch.equal(orc.batched_nms(boxes, scores, idxs, thr), tv.ops.batched_nms(boxes, scores, idxs, thr))


@pytest.mark.parametrize("seed", range(3))
def test_sweep_roi_align_rotated_vs_compiled_reference(seed, golden):
    # inputs and the compiled reference's results stored by make_golden.py (gen_compiled_reference)
    d = golden("compiled_reference")
    ph, pw, sr = (int(v) for v in d[f"sweep{seed}_cfg"])
    x, rois, ref, go, gref = (T(d[f"sweep{seed}_{k}"]) for k in ("x", "rois", "y", "go", "gx"))
    n, c, h, w = x.shape
    assert torch.allclose(orc.roi_align_rotated_forward(x, rois, 0.25, ph, pw, sr), ref, rtol=1e-4, atol=1e-5)
    assert torch.allclose(orc.roi_align_rotated_backward(go, rois, 0.25, ph, pw, n, c, h, w, sr), gref, rtol=1e-4, atol=1e-4)
