#!/usr/bin/env python
"""bench.py -- throughput of the detection hot path at BASELINE.json configs[2] (the config the metric is quoted on).

One "step" = one pass of the per-GPU custom-op hot path of a Mask R-CNN R50-FPN TRAINING iteration with 2 images per GPU
(synthetic 3x800x1333 images -> padded 800x1344, FPN p2..p5 256 ch fp32), forward AND backward of every op:

    rpn_nms     2 x batched_nms(8819 boxes, 5 levels, thr 0.7)                     (proposal_utils.py:121, one per image)
    box_pool    ROIPooler 7x7 aligned, 1024 RoIs (512 / image)  fwd + bwd          (roi_heads.py:798 -> poolers.py:206)
    mask_pool   ROIPooler 14x14, 256 foreground RoIs (128 / image)  fwd + bwd      (roi_heads.py:843)
    dconv       the 13 DeformConv 3x3 layers of the R50 dconv c3-c5 variant, fwd + bwd (input, offset, weight grads):
                4 x C=128 @100x168, 6 x C=256 @50x84, 3 x C=512 @25x42             (backbone/resnet.py:213-329)

The backbone / heads between those ops are cuDNN / cuBLAS work outside the scope of this repository (DESIGN.md).  The
step is captured in CUDA graphs; before timing, its outputs are checked once against the oracle.  The inference hot path
of configs[1] (last round's headline) is kept as `extra.inference_hot_path`.  Prints ONE JSON line (DESIGN.md section 5).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned (rank 0) as DIR/<name>.npy, so that two builds can be compared
output for output on the same seeded inputs (see dump_step_outputs).
"""
import argparse
import json
import math
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

IMG_H, IMG_W = 800, 1333
PAD_H, PAD_W = 800, 1344
LEVELS = [(200, 336, 1 / 4), (100, 168, 1 / 8), (50, 84, 1 / 16), (25, 42, 1 / 32)]
C = 256
IMGS_PER_GPU = 2
N_RPN_TRAIN = 8819      # 2000 per level p2..p5 + 819 on p6 (pre_nms_topk 2000 in training)
N_BOX_ROIS = 512        # per image (ROI_HEADS.BATCH_SIZE_PER_IMAGE)
N_MASK_ROIS = 128       # per image (foreground quarter)
DCONV_STAGES = [(128, 100, 168, 4), (256, 50, 84, 6), (512, 25, 42, 3)]   # (channels, H, W, layers): R50 res3..res5
# inference hot path (configs[1]), reported under `extra`
N_PROPOSALS = 1000
N_RPN_BOXES = 4819
N_DET_CANDIDATES = 3000
N_DET = 100
MASK_SIDE = 28
METRIC = "Mask R-CNN R50-FPN training hot-path images/sec (custom-op path fwd+bwd, 2 images/GPU)"
WORKLOAD = ("configs[2]: Mask R-CNN R50-FPN training hot path, 2 synthetic 3x800x1333 images per GPU: 2 x RPN batched_nms "
            "(8819 boxes), box ROIPooler fwd+bwd (1024 RoIs, 7x7), mask ROIPooler fwd+bwd (256 RoIs, 14x14), 13 DeformConv "
            "layers of the R50 dconv c3-c5 variant fwd+bwd; fp32 tensors, deform-conv contraction in bf16x3 on tcgen05")


# ----------------------------------------------------------------------------------------- synthetic inputs
def synth_boxes(g, n, smin=16.0, smax=600.0):
    """sqrt(area) log-uniform in [16,600] px, aspect log-uniform in [1/2,2], centres uniform, clipped (SURVEY 8d)."""
    s = torch.exp(torch.rand(n, generator=g) * (math.log(smax) - math.log(smin)) + math.log(smin))
    a = torch.exp((torch.rand(n, generator=g) - 0.5) * 2 * math.log(2.0))
    w, h = s * torch.sqrt(a), s / torch.sqrt(a)
    cx, cy = torch.rand(n, generator=g) * IMG_W, torch.rand(n, generator=g) * IMG_H
    b = torch.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1)
    b[:, 0::2].clamp_(0, IMG_W)
    b[:, 1::2].clamp_(0, IMG_H)
    return b


def make_image_inputs(seed):
    """One image of the inference hot path (configs[1]); also used by tools/ and the `extra` line."""
    g = torch.Generator().manual_seed(seed)
    d = {}
    d["feats"] = [torch.randn(1, C, h, w, generator=g) for (h, w, _) in LEVELS]
    d["rpn_boxes"] = synth_boxes(g, N_RPN_BOXES, 16.0, 500.0)
    d["rpn_scores"] = torch.rand(N_RPN_BOXES, generator=g)
    lv = torch.cat([torch.full((1000,), i) for i in range(4)] + [torch.full((819,), 4)])
    d["rpn_levels"] = lv.to(torch.int64)
    d["proposals"] = synth_boxes(g, N_PROPOSALS)
    # Fast R-CNN candidates: each is a jittered copy of one of ~300 objects so that NMS has real work to do
    base = synth_boxes(g, 300, 24.0, 500.0)
    pick = torch.randint(0, 300, (N_DET_CANDIDATES,), generator=g)
    d["det_boxes"] = (base[pick] + torch.randn(N_DET_CANDIDATES, 4, generator=g) * 6).clamp_(0, IMG_W)
    d["det_boxes"][:, 2:] = torch.maximum(d["det_boxes"][:, 2:], d["det_boxes"][:, :2] + 2)
    d["det_scores"] = 0.05 + 0.95 * torch.rand(N_DET_CANDIDATES, generator=g)
    d["det_classes"] = (pick % 80).to(torch.int64)
    d["masks"] = torch.rand(N_DET, MASK_SIDE, MASK_SIDE, generator=g)
    return d


def make_train_inputs(seed):
    """One training step's inputs of the hot path (2 images): dict of CPU tensors (lists for per-level / per-layer data)."""
    g = torch.Generator().manual_seed(seed)
    n = IMGS_PER_GPU
    d = {}
    d["feats"] = [torch.randn(n, C, h, w, generator=g) for (h, w, _) in LEVELS]
    d["rpn_boxes"] = [synth_boxes(g, N_RPN_TRAIN, 16.0, 500.0) for _ in range(n)]
    d["rpn_scores"] = [torch.rand(N_RPN_TRAIN, generator=g) for _ in range(n)]
    d["rpn_levels"] = torch.cat([torch.full((2000,), i) for i in range(4)] + [torch.full((819,), 4)]).to(torch.int64)
    d["box_rois"] = [synth_boxes(g, N_BOX_ROIS) for _ in range(n)]
    d["mask_rois"] = [b[:N_MASK_ROIS].contiguous() for b in d["box_rois"]]
    d["go_box"] = torch.randn(n * N_BOX_ROIS, C, 7, 7, generator=g)
    d["go_mask"] = torch.randn(n * N_MASK_ROIS, C, 14, 14, generator=g)
    # deformable conv: per stage one (x, offset, grad_out) set shared by the stage's layers, one weight per layer
    d["dc_x"], d["dc_off"], d["dc_go"], d["dc_w"] = [], [], [], []
    for (c, h, w, layers) in DCONV_STAGES:
        d["dc_x"].append(torch.randn(n, c, h, w, generator=g))
        d["dc_off"].append(torch.randn(n, 18, h, w, generator=g) * 2)
        d["dc_go"].append(torch.randn(n, c, h, w, generator=g))
        d["dc_w"].append([torch.randn(c, c, 3, 3, generator=g) * (1.0 / math.sqrt(9 * c)) for _ in range(layers)])
    return d


def tensors_of(d):
    for v in d.values():
        if isinstance(v, torch.Tensor):
            yield v
        else:
            for t in v:
                if isinstance(t, torch.Tensor):
                    yield t
                else:
                    yield from t


# constants read off the committed ncu --set full capture of this step (profiles/r2_ncu_full.txt); sm__pipe_tensor_cycles_active
# per kernel, res3 (C=128) / res4 (C=256) / res5 (C=512) layers
R2_NCU = {"bwd_pair_dram_bytes": 57178624 + 99328 + 172992256 + 4922624,
          "tensor_pipe_active_pct": {"dcn_fwd_tc_kernel": [16.0, 32.4, 40.0], "dcn_bwd_data_tc_kernel": [8.8, 17.5, 31.8],
                                     "dcn_bwd_weight_cols_kernel": [44.6, 47.8, 51.2]}}

E2E_HALF_KEYS = ("feats", "go_box", "go_mask", "dc_x", "dc_off", "dc_go")  # activations / gradients: bf16 under autocast


def nbytes_of(d, skip=()):
    return sum(t.numel() * t.element_size() for k, v in d.items() if k not in skip for t in tensors_of({k: v}))


def map_tensors(d, fn):
    out = {}
    for k, v in d.items():
        if isinstance(v, torch.Tensor):
            out[k] = fn(v)
        else:
            out[k] = [fn(t) if isinstance(t, torch.Tensor) else [fn(u) for u in t] for t in v]
    return out


def roi_align_algorithmic_bytes(rois_by_image, ph, pw, n_img):
    """SURVEY 8(d): sum_l min(N*C*H_l*W_l, sum_k C*fp_k)*4 + K*C*PH*PW*4 + K*5*4, fp_k = pixel footprint on its level."""
    total, k = 0, 0
    per_level_fp = [0] * len(LEVELS)
    for b in rois_by_image:
        sizes = torch.sqrt((b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1]))
        lv = torch.floor(4 + torch.log2(sizes / 224 + 1e-8)).clamp(2, 5).long() - 2
        for l, (h, w, s) in enumerate(LEVELS):
            bl = b[lv == l] * s - 0.5
            if len(bl):
                fp = (torch.floor(bl[:, 2]) - torch.floor(bl[:, 0]) + 2).clamp(1, w) * \
                     (torch.floor(bl[:, 3]) - torch.floor(bl[:, 1]) + 2).clamp(1, h)
                per_level_fp[l] += int(fp.sum().item())
        k += len(b)
    for l, (h, w, _) in enumerate(LEVELS):
        total += min(n_img * C * h * w, per_level_fp[l] * C) * 4
    return total + k * C * ph * pw * 4 + k * 5 * 4


def roi_align_bwd_algorithmic_bytes(k, ph, pw, n_img):
    """SURVEY 8(d): read grad_out once + write every grad_input byte once (includes the zero fill)."""
    return k * C * ph * pw * 4 + sum(n_img * C * h * w * 4 for (h, w, _) in LEVELS)


def dconv_flops(c, h, w, n):
    return 2.0 * n * c * c * 9 * h * w


def dconv_bwd_algorithmic_bytes(c, h, w, n):
    """SURVEY 8(d): B_fwd = x + offset + weight + out;  bwd ~ 2*B_fwd + x."""
    x, off, wt, out = n * c * h * w * 4, n * 18 * h * w * 4, c * c * 9 * 4, n * c * h * w * 4
    return 2 * (x + off + wt + out) + x


# ----------------------------------------------------------------------------------------- our arm
class TrainRunner:
    """The training hot path on our kernels.  `step` calls the forward / backward custom ops explicitly (what autograd
    would dispatch) so that the whole step is capturable in one CUDA graph; `step_autograd` goes through the public
    detectron2.layers-shaped API and torch.autograd (used by the end-to-end measurement)."""

    def __init__(self, device):
        import detectron2_b200.layers as L
        from detectron2_b200 import ops
        from detectron2_b200.poolers import ROIPooler, convert_boxes_to_pooler_format

        self.L, self.ops, self.dev = L, ops, device
        self.to_rois = convert_boxes_to_pooler_format
        self.scales = [s for (_, _, s) in LEVELS]
        self.box_pooler = ROIPooler(7, self.scales, 0, "ROIAlignV2")
        self.mask_pooler = ROIPooler(14, self.scales, 0, "ROIAlignV2")
        self.shapes = [IMGS_PER_GPU, C] + [v for (h, w, _) in LEVELS for v in (h, w)]

    def to_device(self, d):
        return map_tensors(d, lambda t: t.to(self.dev, non_blocking=True))

    # -- stages (explicit ops: graph-capturable, no autograd bookkeeping)
    def rpn_nms(self, d):
        # one call per image like the reference's loop (the two images' NMS in ONE call, `batched_nms_images_fixed`, measured
        # slower on this step: 281 vs 254 us -- the kernels are latency chains per category, not throughput-bound)
        return [self.L.batched_nms_fixed(b, s, d["rpn_levels"], 0.7) for b, s in zip(d["rpn_boxes"], d["rpn_scores"])]

    def pool_fwd(self, d, which, feats=None):
        ops = self.ops
        out = 7 if which == "box" else 14
        rois = self.to_rois(d[which + "_rois"])
        return ops.roi_pooler_op(feats if feats is not None else d["feats"], rois, self.scales, out, out, 0, True, 2, 5, 4,
                                 224.0), rois

    def pool_bwd(self, d, which, rois, channels_last=False):
        out = 7 if which == "box" else 14
        return self.ops.roi_pooler_backward_op(d["go_" + which], rois, self.shapes, self.scales, out, out, 0, True, 2, 5, 4,
                                               224.0, channels_last)

    def dconv_fwd(self, d, si, li, prec=-1):
        """(y, x_saved, cols): the training forward keeps the channels-last copy of x it ran on and its sampled columns."""
        return self.ops.deform_conv_train_op(d["dc_x"][si], d["dc_off"][si], None, d["dc_w"][si][li], None, [1, 1], [1, 1],
                                             [1, 1], 1, 1, prec)

    def dconv_bwd(self, d, si, li, saved=None, prec=-1):
        """All gradients; `saved` = dconv_fwd's result (what autograd keeps between the two calls)."""
        x, cols = d["dc_x"][si], None
        if saved is not None:
            x = saved[1] if saved[1].numel() else x
            cols = saved[2] if saved[2].numel() else None
        return self.ops.deform_conv_backward_op(x, d["dc_off"][si], None, d["dc_w"][si][li], d["dc_go"][si],
                                                [1, 1], [1, 1], [1, 1], 1, 1, False, True, True, prec, cols)

    def step(self, d):
        ops = self.ops
        outs = {"keep": self.rpn_nms(d)}
        # both heads pool the same pyramid: ONE layout-change launch, the channels-last kernels run in place on it, their
        # channels-last gradients are summed (what autograd's accumulation does) and go back to NCHW in ONE launch
        cl = ops.pyramid_to_channels_last(d["feats"])
        yb, rb = self.pool_fwd(d, "box", cl)
        ym, rm = self.pool_fwd(d, "mask", cl)
        gb = self.pool_bwd(d, "box", rb, True)
        gm = self.pool_bwd(d, "mask", rm, True)
        gsum = [(a + b).permute(0, 2, 3, 1) for a, b in zip(gb, gm)]  # NHWC storage
        outs.update(box=yb, mask=ym, gfeat=ops._from_nhwc(gsum, IMGS_PER_GPU, C, d["go_box"].device))
        outs["dc"] = []
        for si, (_, _, _, layers) in enumerate(DCONV_STAGES):
            for li in range(layers):
                saved = self.dconv_fwd(d, si, li)
                outs["dc"].append((saved[0], self.dconv_bwd(d, si, li, saved)))
        return outs

    # our own kernels per step (torch's add / cat / fill / memset launches not counted; tools/kernel_times.py lists them all)
    KERNELS_PER_STEP = (2 * 3            # NMS: rank, mask, scan (+ compaction in the last CTA)
                        + 1 + 2          # pyramid layout change, channels-last pooler forward per head
                        + 2 * 2 + 1      # per head: zero fill + channels-last pooler backward; gradient layout change back to NCHW
                        + 13 * (3 + 6))  # deform conv fwd: layout, weight tiles, K1 (saves x channels-last + its columns);
    #                                      bwd: zero fill, grad_out tiles, W^T tiles, K2, K3 from the saved columns, weight-gradient re-layout

    def step_autograd(self, d, fixed_nms=False):
        """Public API + torch.autograd: what a training loop runs.  Returns a small result vector (checksums)."""
        L = self.L
        nms = L.batched_nms_fixed if fixed_nms else L.batched_nms  # fixed: padded keep list + device count, no host sync
        for b, s in zip(d["rpn_boxes"], d["rpn_scores"]):
            nms(b, s, d["rpn_levels"], 0.7)
        feats = [f.requires_grad_(True) for f in d["feats"]]
        yb = self.box_pooler(feats, d["box_rois"])
        ym = self.mask_pooler(feats, d["mask_rois"])
        torch.autograd.backward([yb, ym], [d["go_box"], d["go_mask"]])
        sums = [f.grad.sum() for f in feats]
        for f in feats:
            f.grad = None
        for si, (_, _, _, layers) in enumerate(DCONV_STAGES):
            x, off = d["dc_x"][si].requires_grad_(True), d["dc_off"][si].requires_grad_(True)
            for li in range(layers):
                w = d["dc_w"][si][li].requires_grad_(True)
                y = L.deform_conv(x, off, w, 1, 1, 1, 1, 1)
                y.backward(d["dc_go"][si])
                sums.append(w.grad.sum())
                w.grad = None
            sums.append(x.grad.sum())
            x.grad = off.grad = None
        return torch.stack([v.float() for v in sums])


def validate_step(runner, d_host, d_dev, outs):
    """One-off check of the step's outputs against the oracle (CPU restatement) before anything is timed."""
    from oracle import oracle as orc

    orc.load_reference()
    rep = {}
    # NMS of image 0: bit-exact kept indices
    total = 0
    for i, (keep, num) in enumerate(outs["keep"]):  # every image's kept indices, bit-exact
        kept = keep[: int(num.item())].cpu()
        ref = orc.batched_nms(d_host["rpn_boxes"][i], d_host["rpn_scores"][i], d_host["rpn_levels"], 0.7)
        assert torch.equal(kept, ref), "rpn_nms differs from the oracle (image %d)" % i
        total += int(kept.numel())
    rep["rpn_nms_kept"] = total
    # poolers: 48 sampled RoIs (forward, all channels) and the first 4 channels of the feature gradient (the op is
    # independent per channel, so the oracle runs on 4-channel slices of the same inputs)
    for which, out, yk in (("box", 7, "box"), ("mask", 14, "mask")):
        per_img = d_host[which + "_rois"]
        rois = torch.cat([torch.cat([torch.full((len(b), 1), float(i)), b], 1) for i, b in enumerate(per_img)])
        sizes = torch.sqrt((rois[:, 3] - rois[:, 1]) * (rois[:, 4] - rois[:, 2]))
        lv = torch.floor(4 + torch.log2(sizes / 224 + 1e-8)).clamp(2, 5).long() - 2
        sel = torch.arange(0, len(rois), max(1, len(rois) // 48))
        y = outs[yk].cpu()
        for l, (_, _, s) in enumerate(LEVELS):
            idx = sel[lv[sel] == l]
            if len(idx):
                r = orc.roi_align_forward(d_host["feats"][l], rois[idx], s, out, out, 0, True)
                err = (y[idx] - r).abs().max().item()
                assert err <= 1e-4 * r.abs().max().item() + 1e-5, ("pooler fwd", which, l, err)
    gsum = [torch.zeros(IMGS_PER_GPU, 4, h, w) for (h, w, _) in LEVELS]
    for which, out in (("box", 7), ("mask", 14)):
        per_img = d_host[which + "_rois"]
        rois = torch.cat([torch.cat([torch.full((len(b), 1), float(i)), b], 1) for i, b in enumerate(per_img)])
        sizes = torch.sqrt((rois[:, 3] - rois[:, 1]) * (rois[:, 4] - rois[:, 2]))
        lv = torch.floor(4 + torch.log2(sizes / 224 + 1e-8)).clamp(2, 5).long() - 2
        go = d_host["go_" + which][:, :4].contiguous()
        for l, (h, w, s) in enumerate(LEVELS):
            idx = torch.nonzero(lv == l, as_tuple=True)[0]
            if len(idx):
                gsum[l] += orc.roi_align_backward(go[idx], rois[idx], s, out, out, IMGS_PER_GPU, 4, h, w, 0, True)
    for l in range(len(LEVELS)):
        got = outs["gfeat"][l][:, :4].cpu()
        err = (got - gsum[l]).abs().max().item()
        assert err <= 1e-4 * gsum[l].abs().max().item() + 2e-4, ("pooler bwd", l, err)
    rep["pooler_bwd_checked_channels"] = 4
    # deform conv: the tensor-core results of one layer per stage against the fp32 FFMA path (itself pinned to the
    # oracle by tests/test_gpu_parity.py) and, for the res5 layer, against the oracle on the first image
    k = 0
    for si, (c, h, w, layers) in enumerate(DCONV_STAGES):
        y, (gx, goff, _, gw, _) = outs["dc"][k]
        y0 = runner.dconv_fwd(d_dev, si, 0, 0)[0]
        g0 = runner.dconv_bwd(d_dev, si, 0, None, 0)
        for name, a, b in (("y", y, y0), ("gx", gx, g0[0]), ("goff", goff, g0[1]), ("gw", gw, g0[3])):
            err = (a - b).abs().max().item()
            assert err <= 1e-4 * b.abs().max().item() + 1e-6, ("dconv", si, name, err)
        k += layers
    si = 2
    r = orc.deform_conv_forward(d_host["dc_x"][si][:1], d_host["dc_off"][si][:1], None, d_host["dc_w"][si][0], None, 1, 1, 1, 1, 1)
    got = outs["dc"][10][0][:1].cpu()
    err = (got - r).abs().max().item()
    assert err <= 1e-4 * r.abs().max().item() + 1e-6, ("dconv vs oracle", err)
    rep["dconv_vs_oracle_max_abs_err"] = err
    return rep


DUMP_SAMPLE = 1 << 17  # elements stored of a larger output


def dump_step_outputs(outs, out_dir):
    """Write the outputs of one TrainRunner.step as out_dir/<name>.npy: floating-point outputs in float32, kept indices and
    counts in float64 (exact).  An output of more than DUMP_SAMPLE elements is stored as the 1-D sample of DUMP_SAMPLE
    elements at fixed positions of its flattened (logical, row-major) order: torch.randperm with seed 0, sorted.  The
    positions depend only on the output's size, so every build stores the same elements.  Returns the bytes written."""
    import numpy as np

    arrays = {}
    for i, (keep, num) in enumerate(outs["keep"]):
        arrays["rpn_nms_keep_img%d" % i] = keep[: int(num.item())]
        arrays["rpn_nms_num_kept_img%d" % i] = num
    arrays["box_pool_fwd"], arrays["mask_pool_fwd"] = outs["box"], outs["mask"]
    for l, g in enumerate(outs["gfeat"]):
        arrays["feature_grad_p%d" % (l + 2)] = g
    k = 0
    for c, _, _, layers in DCONV_STAGES:
        for li in range(layers):
            y, (gx, goff, _, gw, _) = outs["dc"][k]
            for name, t in (("out", y), ("grad_x", gx), ("grad_offset", goff), ("grad_weight", gw)):
                arrays["dconv_c%d_layer%d_%s" % (c, li, name)] = t
            k += 1
    os.makedirs(out_dir, exist_ok=True)
    total, positions = 0, {}
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            if t.numel() not in positions:
                perm = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))
                positions[t.numel()] = perm[:DUMP_SAMPLE].sort().values.to(t.device)
            t = t.reshape(-1)[positions[t.numel()]]
        a = t.cpu().numpy().astype(np.float32 if t.is_floating_point() else np.float64)
        np.save(os.path.join(out_dir, name + ".npy"), a)
        total += a.nbytes
    assert total <= 64 << 20, total
    return total


# ----------------------------------------------------------------------------------------- inference hot path (extra)
class InferenceRunner:
    def __init__(self, device):
        import detectron2_b200.layers as L
        from detectron2_b200.poolers import ROIPooler, pyramid_to_channels_last

        self.to_channels_last = pyramid_to_channels_last
        self.L, self.dev = L, device
        scales = [s for (_, _, s) in LEVELS]
        self.box_pooler = ROIPooler(7, scales, 0, "ROIAlignV2")
        self.mask_pooler = ROIPooler(14, scales, 0, "ROIAlignV2")

    def step(self, d):
        L = self.L
        keep, nk = L.batched_nms_fixed(d["rpn_boxes"], d["rpn_scores"], d["rpn_levels"], 0.7)
        feats = self.to_channels_last(d["feats"])
        box_feats = self.box_pooler(feats, [d["proposals"]])
        dk, nd = L.batched_nms_fixed(d["det_boxes"], d["det_scores"], d["det_classes"], 0.5)
        pos = torch.arange(N_DET, device=dk.device)
        dk = torch.where(pos < nd, dk[:N_DET], torch.zeros_like(dk[:N_DET]))  # padded slots -> a valid row
        det = d["det_boxes"][dk]
        mask_feats = self.mask_pooler(feats, [det])
        pasted = L.paste_masks_in_image(d["masks"][: det.shape[0]], det, (IMG_H, IMG_W), 0.5)
        return keep, box_feats, det, mask_feats, pasted


# ----------------------------------------------------------------------------------------- reference (CPU) arm
class ReferenceRunner:
    """The reference's own CPU implementation of the same step: torchvision CPU ops (the backend detectron2.layers calls:
    roi_align.py:3,58 / nms.py:5-22 / deform_conv.py:55-57) with torch.autograd, the per-level ROIPooler loop
    (poolers.py:245-263)."""

    def __init__(self):
        import torchvision

        self.tv = torchvision

    def pooler(self, feats, per_img, out, frac):
        tv = self.tv
        boxes = torch.cat([torch.cat([torch.full((max(1, int(len(b) * frac)), 1), float(i)), b[: max(1, int(len(b) * frac))]], 1)
                           for i, b in enumerate(per_img)])
        sizes = torch.sqrt((boxes[:, 3] - boxes[:, 1]) * (boxes[:, 4] - boxes[:, 2]))
        lv = torch.floor(4 + torch.log2(sizes / 224 + 1e-8)).clamp(2, 5).to(torch.int64) - 2
        res = torch.zeros(len(boxes), C, out, out)
        for l, (_, _, s) in enumerate(LEVELS):
            inds = torch.nonzero(lv == l, as_tuple=True)[0]
            res = res.index_put((inds,), tv.ops.roi_align(feats[l], boxes[inds], (out, out), s, 0, True))
        return res

    def step(self, d, frac=1.0):
        tv = self.tv
        n_rpn = max(8, int(N_RPN_TRAIN * frac))
        for b, s in zip(d["rpn_boxes"], d["rpn_scores"]):
            tv.ops.boxes.batched_nms(b[:n_rpn].float(), s[:n_rpn], d["rpn_levels"][:n_rpn], 0.7)
        feats = [f.requires_grad_(True) for f in d["feats"]]
        yb = self.pooler(feats, d["box_rois"], 7, frac)
        ym = self.pooler(feats, d["mask_rois"], 14, frac)
        torch.autograd.backward([yb, ym], [d["go_box"][: len(yb)], d["go_mask"][: len(ym)]])
        for f in feats:
            f.grad = None
        # deformable conv: a `frac` share of the 13 layers, taken round-robin over the stages
        order = [(0, 0), (1, 0), (2, 0), (0, 1), (1, 1), (2, 1), (0, 2), (1, 2), (2, 2), (0, 3), (1, 3), (1, 4), (1, 5)]
        n_layers = max(1, int(round(13 * frac)))
        for (si, li) in order[:n_layers]:
            x, off, w = d["dc_x"][si].requires_grad_(True), d["dc_off"][si].requires_grad_(True), d["dc_w"][si][li].requires_grad_(True)
            y = tv.ops.deform_conv2d(x, off, w, None, 1, 1, 1)
            y.backward(d["dc_go"][si])
            x.grad = off.grad = w.grad = None
        return n_layers


def time_reference(steps, warmup, budget_s=150.0):
    ref = ReferenceRunner()
    d = make_train_inputs(0)
    # "all the host threads it can use": torchvision's CPU kernels stop scaling (and then regress) well before 100+
    # threads, so pick the fastest of a few thread counts on a 1/16 sample and report the count actually used.
    ncpu = os.cpu_count() or 1
    best = None
    for nt in sorted({ncpu, min(ncpu, 64), min(ncpu, 32), min(ncpu, 16)}, reverse=True):
        torch.set_num_threads(nt)
        t0 = time.perf_counter()
        ref.step(d, 1 / 16)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, nt)
    t16, nt = best
    torch.set_num_threads(nt)
    frac = 1.0
    while frac > 1 / 64 and (steps + warmup) * t16 * 16 * frac > budget_s:
        frac /= 2
    for _ in range(warmup):
        ref.step(d, frac)
    t0 = time.perf_counter()
    for _ in range(steps):
        ref.step(d, frac)
    dt = time.perf_counter() - t0
    return frac * steps * IMGS_PER_GPU / dt, dt / steps * 1e3, frac, torch.get_num_threads()


# ----------------------------------------------------------------------------------------- multi-GPU aggregation
def image_seeds(rank, nbuf):
    """Synthetic-input seeds of one rank: replicas never share an image (image-parallel sharding, no data-path collective)."""
    return [1000 * rank + i for i in range(nbuf)]


def max_over_ranks(values_ms, dist, device):
    """Element-wise MAX over ranks of per-rank elapsed times (the only collective of the benchmark)."""
    t = torch.tensor(list(values_ms), dtype=torch.float64, device=device)
    if dist is not None and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.tolist()


def aggregate_throughput(world, steps, elapsed_ms, images_per_step=IMGS_PER_GPU):
    """Whole-job images/s: every rank processed `steps` steps of `images_per_step` images in (max over ranks) elapsed_ms."""
    return world * steps * images_per_step / (elapsed_ms / 1e3)


def pin_to_local_cpus(local_rank, world):
    """Spread the ranks' host threads (pinned-memory copies, launches) over the CPU set this process is allowed to use,
    one contiguous block per rank: without it 8 ranks' H2D/D2H staging contend for the same cores / NUMA node."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
        if world > 1 and len(cpus) >= 2 * world:
            per = len(cpus) // world
            os.sched_setaffinity(0, set(cpus[local_rank * per:(local_rank + 1) * per]))
            return per
    except (AttributeError, OSError):
        pass
    return None


# ----------------------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.active = False  # samples are only kept while a timed region is running

    def run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                if self.active:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
                time.sleep(0.005)
        except Exception as e:  # NVML unavailable: report that instead of inventing clocks
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "samples": len(s),
                "reasons": sorted(self.reasons)}


def graph_of(fn, stream):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(stream):
        with torch.cuda.graph(g, stream=stream):
            keep = fn()
    return g, keep


def time_graphs(graphs, reps):
    """Mean device time (ms) of one replay, rotating over the graphs (one per input set)."""
    for i in range(3):
        graphs[i % len(graphs)].replay()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for i in range(reps):
        graphs[i % len(graphs)].replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


# ----------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (rank 0, impl ours) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    base = {"metric": METRIC, "unit": "img/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "images_per_gpu": IMGS_PER_GPU, "rpn_boxes_per_image": N_RPN_TRAIN,
                       "box_rois": IMGS_PER_GPU * N_BOX_ROIS, "mask_rois": IMGS_PER_GPU * N_MASK_ROIS, "dconv_layers": 13,
                       "parallelism": "replicas (image-parallel, no data-path collective)"}}

    if args.impl == "reference":
        if rank != 0:
            return
        v, ms, frac, cores = time_reference(args.steps, max(args.warmup, 1))
        line = dict(base)
        line.update({"impl": "reference", "value": v, "ms_per_step": ms, "n_gpus": args.gpus,
                     "cpu_baseline": {"value": v, "unit": "img/s", "cores": cores, "kind": "reference",
                                      "sample": "%.4g of one training step's hot path per step (torchvision CPU batched_nms, "
                                                "roi_align fwd+bwd in the reference's per-level ROIPooler loop, deform_conv2d "
                                                "fwd+bwd with torch.autograd), %d threads" % (frac, cores)},
                     "e2e": {"value": v, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                     "gpu_launches": 0})
        print(json.dumps(line))
        return

    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a CUDA device"
    cpus_per_rank = pin_to_local_cpus(local_rank, world)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)
    sampler = ClockSampler(local_rank)
    sampler.start()  # started before warm-up so that NVML is initialised when the timed region begins
    runner = TrainRunner(dev)
    NBUF = 2  # two input sets: 2 x 183 MB of features + 183 MB of gradients written per step, far beyond the 126 MB L2
    host = [make_train_inputs(sd) for sd in image_seeds(rank, NBUF)]
    devin = [runner.to_device(h) for h in host]
    torch.cuda.synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- correctness of the step, once, before anything is timed
    outs0 = runner.step(devin[0])
    torch.cuda.synchronize()
    validation = validate_step(runner, host[0], devin[0], outs0)
    del outs0

    # ---------------- device-resident throughput ("value"): the whole step captured in CUDA graphs
    for i in range(max(args.warmup, 3)):
        runner.step(devin[i % NBUF])
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    graphs, graph_outs = [], []
    for b in range(NBUF):
        gph, keepalive = graph_of(lambda b=b: runner.step(devin[b]), side)
        graphs.append(gph)
        graph_outs.append(keepalive)
    torch.cuda.synchronize()
    for i in range(max(args.warmup, 3)):
        graphs[i % NBUF].replay()
    barrier()
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.active = True
    t_start.record()
    for i in range(args.steps):
        graphs[i % NBUF].replay()
    t_end.record()
    barrier()
    sampler.active = False
    elapsed_ms = t_start.elapsed_time(t_end)
    if args.dump_outputs and rank == 0:
        # the last timed replay was graphs[(steps - 1) % NBUF]; its outputs live in that graph's static buffers
        dump_step_outputs(graph_outs[(args.steps - 1) % NBUF], args.dump_outputs)
    del graphs, graph_outs

    # ---------------- per-stage device time: each stage captured alone in its own graphs, rotating inputs
    rois_box = [runner.to_rois(d["box_rois"]) for d in devin]
    rois_mask = [runner.to_rois(d["mask_rois"]) for d in devin]
    cls = [runner.ops.pyramid_to_channels_last(d["feats"]) for d in devin]
    gcl = [[torch.zeros(IMGS_PER_GPU, h, w, C, device=dev) for (h, w, _) in LEVELS] for _ in devin]
    stages = {
        "rpn_nms": lambda b: runner.rpn_nms(devin[b]),
        "pyramid_to_channels_last": lambda b: runner.ops.pyramid_to_channels_last(devin[b]["feats"]),
        "box_pool_fwd": lambda b: runner.pool_fwd(devin[b], "box", cls[b]),
        "box_pool_bwd": lambda b: runner.pool_bwd(devin[b], "box", rois_box[b], True),
        "mask_pool_fwd": lambda b: runner.pool_fwd(devin[b], "mask", cls[b]),
        "mask_pool_bwd": lambda b: runner.pool_bwd(devin[b], "mask", rois_mask[b], True),
        "grads_to_nchw": lambda b: runner.ops._from_nhwc(gcl[b], IMGS_PER_GPU, C, dev),
    }
    saved = [[[runner.dconv_fwd(d, si, li) for li in range(layers)] for si, (_, _, _, layers) in enumerate(DCONV_STAGES)]
             for d in devin]
    for si, (c, h, w, layers) in enumerate(DCONV_STAGES):
        stages["dconv_c%d_fwd_x%d" % (c, layers)] = lambda b, si=si, layers=layers: [runner.dconv_fwd(devin[b], si, li) for li in range(layers)]
        stages["dconv_c%d_bwd_x%d" % (c, layers)] = lambda b, si=si, layers=layers: [
            runner.dconv_bwd(devin[b], si, li, saved[b][si][li]) for li in range(layers)]
    stage_ms = {}
    for name, fn in stages.items():
        sg = [graph_of(lambda b=b: fn(b), side) for b in range(NBUF)]
        torch.cuda.synchronize()
        stage_ms[name] = time_graphs([g for g, _ in sg], 10)
        del sg

    # ---------------- end to end through the public API with HOST buffers
    # Every step copies ITS OWN inputs from pinned host memory (feature maps, boxes, head gradients, deform-conv
    # activations and weights) and reads the step's result vector back; a copy stream runs one step ahead of the compute.
    # Two transports are measured: "bf16" -- activations and gradients cross PCIe as bf16, which is what the bf16-autocast
    # training of configs[2] hands these ops (boxes, scores and the fp32 master weights stay fp32; the ops compute in fp32
    # and return the input dtype, like the reference under autocast) -- and "fp32" (every tensor fp32, last round's setup).
    compute_stream = torch.cuda.current_stream()
    h2d_stream = torch.cuda.Stream()

    def e2e_measure(transport, graphed):
        half = transport == "bf16"

        def conv(h):
            to_half = lambda t: t.to(torch.bfloat16) if t.is_floating_point() else t  # noqa: E731
            return {k: map_tensors({k: v}, to_half if (half and k in E2E_HALF_KEYS) else (lambda t: t))[k] for k, v in h.items()}

        hosts = [conv(h) for h in host]
        pinned = [map_tensors(h, lambda t: t.pin_memory()) for h in hosts]
        ring = [runner.to_device(h) for h in hosts]
        h2d_done = [torch.cuda.Event() for _ in range(NBUF)]
        compute_done = [torch.cuda.Event() for _ in range(NBUF)]
        res_host = [torch.empty(4 + 13 + 3, dtype=torch.float32).pin_memory() for _ in range(NBUF)]
        torch.cuda.synchronize()
        step_graphs, step_results = [], []
        if graphed:
            # the public-API step (layers + torch.autograd) of every ring slot captured ONCE in a CUDA graph and replayed per
            # step, the standard whole-step capture of a PyTorch training loop: the step's ~200 launches cost one host call
            for slot in range(NBUF):
                runner.step_autograd(ring[slot], True)  # warm-up on the capture inputs (allocations, opt-ins)
            torch.cuda.synchronize()
            for slot in range(NBUF):
                gph, res = graph_of(lambda slot=slot: runner.step_autograd(ring[slot], True), side)
                step_graphs.append(gph)
                step_results.append(res)
            torch.cuda.synchronize()

        def enqueue_h2d(i):
            slot = i % NBUF
            with torch.cuda.stream(h2d_stream):
                h2d_stream.wait_event(compute_done[slot])
                for src, dst in zip(tensors_of(pinned[slot]), tensors_of(ring[slot])):
                    dst.detach().copy_(src, non_blocking=True)
                h2d_done[slot].record(h2d_stream)

        def e2e_run(n):
            for slot in range(NBUF):
                compute_done[slot].record(compute_stream)
            enqueue_h2d(0)
            for i in range(n):
                slot = i % NBUF
                if i + 1 < n:
                    enqueue_h2d(i + 1)
                compute_stream.wait_event(h2d_done[slot])
                if graphed:
                    step_graphs[slot].replay()
                    res = step_results[slot]
                else:
                    res = runner.step_autograd(ring[slot])
                res_host[slot].copy_(res, non_blocking=True)
                compute_done[slot].record(compute_stream)
            torch.cuda.synchronize()

        e2e_run(2)
        check = res_host[1].clone()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        steps = max(4, args.steps // 2)
        e0.record()
        t_host0 = time.perf_counter()
        e2e_run(steps)
        ms_host = (time.perf_counter() - t_host0) * 1e3
        e1.record()
        barrier()
        del step_graphs, step_results
        # device-event time; the host clock guards against stream-order artefacts
        return max(e0.elapsed_time(e1), ms_host), steps, nbytes_of(hosts[0]), check

    def e2e_measure_graphed(transport):
        """Graph replay of the public-API step; if the capture fails, the same measurement with eager launches (never lose the
        bench line to a capture problem).  A failed capture raises before the measurement's first barrier, so every rank runs
        the same number of barriers whichever way it goes."""
        try:
            return e2e_measure(transport, True) + (True,)
        except Exception as exc:
            sys.stderr.write("graphed end-to-end step (%s) failed (%s: %s); measuring eagerly\n" % (transport, type(exc).__name__, exc))
            torch.cuda.synchronize()
            return e2e_measure(transport, False) + (False,)

    e2e_ms, e2e_steps, e2e_bytes, chk_half, e2e_graphed = e2e_measure_graphed("bf16")
    e2e32_ms, e2e32_steps, e2e32_bytes, chk_full, _ = e2e_measure_graphed("fp32")
    e2e_eager_ms, e2e_eager_steps, _, chk_eager = e2e_measure("fp32", False)
    assert torch.allclose(chk_eager, chk_full, rtol=1e-3, atol=1e-3 * chk_full.abs().max().item()), "graphed step differs from eager"
    # the two transports run the same step: their result vectors (gradient checksums of slot 1) agree to bf16 rounding
    scale_ref = chk_full.abs().max().item()
    e2e_dev = (chk_half - chk_full).abs().max().item() / max(scale_ref, 1e-30)
    assert e2e_dev < 5e-2, ("bf16-transport step disagrees with the fp32 step", e2e_dev)

    # ---------------- extra: the inference hot path of configs[1] (last round's headline), graph-captured
    inf_ms = None
    try:
        inf = InferenceRunner(dev)
        ihost = [make_image_inputs(sd) for sd in image_seeds(rank, 3)]
        idev = [map_tensors(h, lambda t: t.to(dev)) for h in ihost]
        for b in range(3):
            inf.step(idev[b])
        torch.cuda.synchronize()
        ig = [graph_of(lambda b=b: inf.step(idev[b]), side) for b in range(3)]
        torch.cuda.synchronize()
        inf_ms = time_graphs([g for g, _ in ig], 30)
        del ig, idev
    except Exception as e:  # supplementary only: never hide the headline numbers
        inf_ms = "failed: %s" % type(e).__name__

    sampler.stop_flag = True
    elapsed_ms, e2e_ms, e2e32_ms, e2e_eager_ms = max_over_ranks([elapsed_ms, e2e_ms, e2e32_ms, e2e_eager_ms], dist, dev)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    value = aggregate_throughput(world, args.steps, elapsed_ms)
    e2e_value = aggregate_throughput(world, e2e_steps, e2e_ms)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = peaks.get("hbm_gbs", 6650.0)
    tf_peak = peaks.get("bf16_tflops_sustained", 1400.0)  # the kernel is timed inside a long step
    src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    # dominant kernels of the step: the deform-conv backward of the res3 stage (4 layers of 2 x 128 x 100 x 168)
    c, h, w, layers = DCONV_STAGES[0]
    bwd_ms = stage_ms["dconv_c128_bwd_x4"] / layers
    flops_bwd = 2 * dconv_flops(c, h, w, IMGS_PER_GPU)  # dX-columns GEMM + dW GEMM (SURVEY 8d)
    ach = flops_bwd / (bwd_ms / 1e3) / 1e12
    box_alg_f = roi_align_algorithmic_bytes(host[0]["box_rois"], 7, 7, IMGS_PER_GPU)
    box_alg_b = roi_align_bwd_algorithmic_bytes(IMGS_PER_GPU * N_BOX_ROIS, 7, 7, IMGS_PER_GPU)

    def gbs(nbytes, ms):
        return nbytes / (ms / 1e3) / 1e9

    line = dict(base)
    line.update({
        "value": value, "ms_per_step": elapsed_ms / args.steps, "n_gpus": world,
        "e2e": {"value": e2e_value, "unit": "img/s", "h2d_bytes_per_step": e2e_bytes, "d2h_bytes_per_step": 20 * 4,
                "steps": e2e_steps, "graphed": e2e_graphed, "transport": "bf16 activations and gradients (what the bf16-autocast training of configs[2] "
                                                 "hands these ops), fp32 boxes / scores / master weights; fp32 arithmetic inside the ops",
                "pipeline": "public API (detectron2_b200.layers + torch.autograd) captured once per input slot in a CUDA graph and "
                            "replayed; H2D of step i+1 overlaps the compute of step i; every step copies its own inputs from pinned "
                            "host memory and reads its result vector (gradient checksums) back",
                "fp32_transport": {"value": aggregate_throughput(world, e2e32_steps, e2e32_ms), "unit": "img/s",
                                   "h2d_bytes_per_step": e2e32_bytes, "steps": e2e32_steps},
                "fp32_transport_eager": {"value": aggregate_throughput(world, e2e_eager_steps, e2e_eager_ms), "unit": "img/s",
                                         "what": "the same step launched eagerly every iteration (no graph): host-launch-bound"},
                "bf16_vs_fp32_result_rel_dev": e2e_dev},
        "gpu_launches": TrainRunner.KERNELS_PER_STEP * args.steps,
        "clocks": sampler.summary(),
        "stages_ms": {k: round(v, 4) for k, v in stage_ms.items()},
        "validation": validation,
        "l2": "two input sets rotate (2 x 183 MB of feature maps) and every step writes 183 MB of gradients: > 126 MB L2",
        "roofline": {"kernel": "deform-conv backward, R50 res3 layer (2 x 128 x 100 x 168): dcn_bwd_data_tc_kernel + "
                               "dcn_bwd_weight_cols_kernel (+ their operand pre-tiling / zero-fill / re-layout launches)",
                     "bound": "tensor", "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s", "frac": ach / tf_peak,
                     "peak_source": src + ", sustained bf16", "algorithmic_flops": flops_bwd, "avg_launch_ms": bwd_ms,
                     "note": "bf16x3 issues 3 MMAs per algorithmic product (fp32-class accuracy); the data-gradient kernel is bound "
                             "by the L2 vector reductions of its scatter (4 corners x 16 B per 4 channels and kernel point: %.0f MB "
                             "per launch against the 5.9 TB/s red.v4 ceiling of profiles/r2_microbench.txt), see DESIGN.md section 4"
                             % (IMGS_PER_GPU * h * w * 9 * c * 16 / 1e6),
                     "algorithmic_bytes": dconv_bwd_algorithmic_bytes(c, h, w, IMGS_PER_GPU),
                     "achieved_hbm_gbs": gbs(dconv_bwd_algorithmic_bytes(c, h, w, IMGS_PER_GPU), bwd_ms),
                     # DRAM bytes of the two kernels from the committed capture (profiles/r2_ncu_full.txt, launches 11 + 12:
                     # dcn_bwd_data_tc_kernel 57.2 + 0.1 MB, dcn_bwd_weight_cols_kernel 173.0 + 4.9 MB -- the latter streams the
                     # forward's saved columns back, 155 MB by design, instead of sampling x a second time)
                     "traffic": R2_NCU["bwd_pair_dram_bytes"],
                     "tensor_pipe_active_pct_ncu": R2_NCU["tensor_pipe_active_pct"]},
        "roofline_other": {
            "roi_align_fwd_box_pooler": {"bound": "hbm", "algorithmic_bytes": box_alg_f, "avg_launch_ms": stage_ms["box_pool_fwd"],
                                         "achieved": gbs(box_alg_f, stage_ms["box_pool_fwd"]), "peak": hbm, "unit": "GB/s",
                                         "frac": gbs(box_alg_f, stage_ms["box_pool_fwd"]) / hbm,
                                         "includes": "roi_align_nhwc_kernel on the channels-last pyramid (layout change timed separately)"},
            "roi_align_bwd_box_pooler": {"bound": "hbm", "algorithmic_bytes": box_alg_b, "avg_launch_ms": stage_ms["box_pool_bwd"],
                                         "achieved": gbs(box_alg_b, stage_ms["box_pool_bwd"]), "peak": hbm, "unit": "GB/s",
                                         "frac": gbs(box_alg_b, stage_ms["box_pool_bwd"]) / hbm,
                                         "includes": "zero fill + roi_align_bwd_nhwc_kernel (layout change back timed separately)"},
            "deform_conv_fwd_res3": {"bound": "tensor", "avg_launch_ms": stage_ms["dconv_c128_fwd_x4"] / layers,
                                     "achieved": dconv_flops(c, h, w, IMGS_PER_GPU) / (stage_ms["dconv_c128_fwd_x4"] / layers / 1e3) / 1e12,
                                     "peak": tf_peak, "unit": "TFLOP/s",
                                     "frac": dconv_flops(c, h, w, IMGS_PER_GPU) / (stage_ms["dconv_c128_fwd_x4"] / layers / 1e3) / 1e12 / tf_peak},
        },
    })
    line["extra"] = {"inference_hot_path": {"ms_per_image": inf_ms,
                                            "img_s": (1e3 / inf_ms * world) if isinstance(inf_ms, float) else None,
                                            "what": "configs[1] hot path per image (RPN NMS 4819, box pooler 1000 RoIs, detection NMS, "
                                                    "mask pooler 100 RoIs, paste 100 masks), CUDA graph, inputs resident"},
                     "cpus_per_rank": cpus_per_rank}
    if world == 1:
        v, ms, frac, cores = time_reference(2, 1, budget_s=25.0)
        line["cpu_baseline"] = {"value": v, "unit": "img/s", "cores": cores, "kind": "reference",
                                "sample": "2 steps x %.4g of one training step's hot path (torchvision CPU batched_nms, roi_align "
                                          "fwd+bwd in the per-level ROIPooler loop, deform_conv2d fwd+bwd), %d threads" % (frac, cores)}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
