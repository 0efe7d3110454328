"""The `detectron2._C`-shaped deform-conv shim (detectron2_b200/_C.py, SURVEY.md 8b "pybind functions").

CPU part: the calls that the REAL, unmodified reference autograd Functions `_DeformConv` / `_ModulatedDeformConv`
(detectron2/layers/deform_conv.py:29-184, :205-313) make into `detectron2._C` were recorded once from the reference
(tests/golden/reference_shim_protocol.npz, written by tests/golden/make_golden.py) and are replayed here against a module
with our shim's signatures whose five entry points are backed by the CPU oracle: what is verified is the CALL PROTOCOL the
reference uses against our signatures -- argument order (width-first for DCNv1), caller-allocated outputs written in
place, gradients accumulated into zero-initialised buffers -- by comparing the buffers the reference Functions return
with torchvision autograd.  GPU part: the same protocol, restated call by call, against the real kernels.
"""
import inspect
import json
import math
import types

import pytest
import torch


class FakeCuda(torch.Tensor):
    """CPU tensor that claims to live on a GPU (the reference wrappers only test the flag)."""

    @property
    def is_cuda(self):
        return True


def _fc(t):
    return None if t is None else torch.Tensor._make_subclass(FakeCuda, t, t.requires_grad)


def test_reference_functions_drive_the_shim_signatures(golden):
    import torchvision

    from detectron2_b200 import _C as real_shim

    # a module with OUR signatures whose bodies are the CPU oracle (torchvision deform_conv2d + autograd)
    shim = types.ModuleType("detectron2._C")
    calls = []

    def plain(t):
        return None if t is None else t.detach().as_subclass(torch.Tensor)

    def tv_all(x, off, mask, w, bias, stride, pad, dil, go=None):
        with torch.enable_grad():  # the reference's backward runs under once_differentiable (grad mode off)
            xs = [plain(t).clone().requires_grad_(True) if t is not None else None for t in (x, off, mask, w, bias)]
            y = torchvision.ops.deform_conv2d(xs[0], xs[1], xs[3], xs[4], stride, pad, dil, xs[2])
            if go is None:
                return y.detach()
            y.backward(plain(go))
            return [None if t is None else t.grad for t in xs]

    def deform_conv_forward(input, weight, offset, output, columns, ones, kW, kH, dW, dH, padW, padH, dilW, dilH, group,
                            deformable_group, im2col_step):
        calls.append("deform_conv_forward")
        assert (kW, kH) == (weight.shape[3], weight.shape[2]) and group == 1 and deformable_group == 1
        output.copy_(tv_all(input, offset, None, weight, None, (dH, dW), (padH, padW), (dilH, dilW)))
        return 1

    def deform_conv_backward_input(input, offset, gradOutput, gradInput, gradOffset, weight, columns, kW, kH, dW, dH, padW,
                                   padH, dilW, dilH, group, deformable_group, im2col_step):
        calls.append("deform_conv_backward_input")
        assert float(gradInput.abs().sum()) == 0.0 and float(gradOffset.abs().sum()) == 0.0  # zero-initialised by the caller
        g = tv_all(input, offset, None, weight, None, (dH, dW), (padH, padW), (dilH, dilW), gradOutput)
        gradInput.copy_(g[0])
        gradOffset.copy_(g[1])
        return 1

    def deform_conv_backward_filter(input, offset, gradOutput, gradWeight, columns, ones, kW, kH, dW, dH, padW, padH, dilW,
                                    dilH, group, deformable_group, scale, im2col_step):
        calls.append("deform_conv_backward_filter")
        g = tv_all(input, offset, None, gradWeight.new_zeros(gradWeight.shape) + 0 * plain(gradWeight) + plain(W_HOLDER[0]),
                   None, (dH, dW), (padH, padW), (dilH, dilW), gradOutput)
        gradWeight.add_(g[3], alpha=scale)
        return 1

    def modulated_deform_conv_forward(input, weight, bias, ones, offset, mask, output, columns, kernel_h, kernel_w, stride_h,
                                      stride_w, pad_h, pad_w, dilation_h, dilation_w, group, deformable_group, with_bias):
        calls.append("modulated_deform_conv_forward")
        output.copy_(tv_all(input, offset, mask, weight, bias if with_bias else None, (stride_h, stride_w), (pad_h, pad_w),
                            (dilation_h, dilation_w)))

    def modulated_deform_conv_backward(input, weight, bias, ones, offset, mask, columns, grad_input, grad_weight, grad_bias,
                                       grad_offset, grad_mask, grad_output, kernel_h, kernel_w, stride_h, stride_w, pad_h,
                                       pad_w, dilation_h, dilation_w, group, deformable_group, with_bias):
        calls.append("modulated_deform_conv_backward")
        g = tv_all(input, offset, mask, weight, bias if with_bias else None, (stride_h, stride_w), (pad_h, pad_w),
                   (dilation_h, dilation_w), grad_output)
        grad_input.copy_(g[0])
        grad_offset.copy_(g[1])
        grad_mask.copy_(g[2])
        grad_weight.add_(g[3])
        if with_bias:
            grad_bias.add_(g[4])

    W_HOLDER = [None]
    oracle_fns = {f.__name__: f for f in (deform_conv_forward, deform_conv_backward_input, deform_conv_backward_filter,
                                          modulated_deform_conv_forward, modulated_deform_conv_backward)}
    for name, fn in oracle_fns.items():
        # the oracle-backed stand-in has EXACTLY the parameter list of the product's shim function
        assert list(inspect.signature(fn).parameters) == list(inspect.signature(getattr(real_shim, name)).parameters), name
        setattr(shim, name, fn)
    shim.get_cuda_version, shim.has_cuda, shim.get_compiler_version = real_shim.get_cuda_version, real_shim.has_cuda, real_shim.get_compiler_version

    # replay the calls the reference Functions made (tests/golden/make_golden.py, gen_reference_shim_protocol): the same
    # arguments in the same positions, buffers allocated as the caller allocated them (NaN where it used new_empty)
    d = golden("reference_shim_protocol")
    protocol = json.loads(str(d["protocol"]))
    inputs = {k: torch.from_numpy(d[k]) for k in ("x", "off", "mask", "w", "bias", "go")}
    x, off, mask, wt, bias, go = (inputs[k] for k in ("x", "off", "mask", "w", "bias", "go"))
    W_HOLDER[0] = wt
    buffers = {}

    def arg(a):
        if isinstance(a, dict) and "input" in a:
            return _fc(inputs[a["input"]].clone())
        if isinstance(a, dict):
            if a["buffer"] not in buffers:
                fill = 0.0 if a["zero"] else math.nan
                buffers[a["buffer"]] = _fc(torch.full(a["shape"], fill))
            return buffers[a["buffer"]]
        return a

    for call in protocol["calls"]:
        getattr(shim, call["fn"])(*[arg(a) for a in call["args"]])
    assert calls == ["deform_conv_forward", "deform_conv_backward_input", "deform_conv_backward_filter",
                     "modulated_deform_conv_forward", "modulated_deform_conv_backward"]
    # ---- DCNv1 through the reference's _DeformConv
    got = {k: plain(buffers[b]) for k, b in protocol["returns"]["v1"].items()}
    assert torch.allclose(got["y"], tv_all(x, off, None, wt, None, (1, 1), (1, 1), (1, 1)), atol=1e-5)
    ref = tv_all(x, off, None, wt, None, (1, 1), (1, 1), (1, 1), go)
    for k, b in zip(("x", "off", "w"), (ref[0], ref[1], ref[3])):
        assert torch.allclose(got[k], b, atol=1e-5), k
    # ---- DCNv2 through the reference's _ModulatedDeformConv
    got = {k: plain(buffers[b]) for k, b in protocol["returns"]["v2"].items()}
    assert torch.allclose(got["y"], tv_all(x, off, mask, wt, bias, (1, 1), (1, 1), (1, 1)), atol=1e-5)
    ref = tv_all(x, off, mask, wt, bias, (1, 1), (1, 1), (1, 1), go)
    for k, b in zip(("x", "off", "mask", "w", "bias"), ref):
        assert torch.allclose(got[k], b, atol=1e-5), k


def test_shim_exports_the_reference_pybind_names():
    # csrc/vision.cpp:86-102
    from detectron2_b200 import _C

    for name in ["get_compiler_version", "get_cuda_version", "has_cuda", "deform_conv_forward", "deform_conv_backward_input",
                 "deform_conv_backward_filter", "modulated_deform_conv_forward", "modulated_deform_conv_backward"]:
        assert callable(getattr(_C, name)), name
    assert len(inspect.signature(_C.deform_conv_forward).parameters) == 17
    assert len(inspect.signature(_C.deform_conv_backward_input).parameters) == 18
    assert len(inspect.signature(_C.deform_conv_backward_filter).parameters) == 18
    assert len(inspect.signature(_C.modulated_deform_conv_forward).parameters) == 19
    assert len(inspect.signature(_C.modulated_deform_conv_backward).parameters) == 24


@pytest.mark.gpu
@pytest.mark.parametrize("c,co,grp", [(8, 12, 1), (128, 128, 1), (64, 64, 4)])
def test_shim_protocol_on_gpu_vs_oracle(c, co, grp):
    """The call sequence of detectron2/layers/deform_conv.py:43-141 (DCNv1) and :205-295 (DCNv2), restated, on the real
    kernels: caller-allocated outputs, zero-initialised gradient buffers, width-first kernel arguments."""
    from detectron2_b200 import _C
    from oracle import oracle as orc

    dev = "cuda"
    g = torch.Generator().manual_seed(c)
    n, h, w = 2, 13, 17
    x = torch.randn(n, c, h, w, generator=g)
    off = torch.randn(n, 18, h, w, generator=g) * 1.5
    mask = torch.sigmoid(torch.randn(n, 9, h, w, generator=g))
    wt = torch.randn(co, c // grp, 3, 3, generator=g) * (1 / math.sqrt(c // grp * 9))
    bias = torch.randn(co, generator=g)
    go = torch.randn(n, co, h, w, generator=g)
    xd, od, md, wd, bd, gd = [t.to(dev) for t in (x, off, mask, wt, bias, go)]
    bufs = [xd.new_empty(0), xd.new_empty(0)]

    def close(a, b, name):
        scale = b.abs().max().item() + 1e-6
        assert (a.cpu() - b).abs().max().item() <= 1e-4 * scale + 1e-5, name

    # ---- DCNv1: forward (deform_conv.py:43-79), backward (:83-141)
    out = xd.new_empty(n, co, h, w)
    _C.deform_conv_forward(xd, wd, od, out, bufs[0], bufs[1], wd.size(3), wd.size(2), 1, 1, 1, 1, 1, 1, grp, 1, 2)
    close(out, orc.deform_conv_forward(x, off, None, wt, None, 1, 1, 1, grp, 1), "y")
    gi, goff, gw = torch.zeros_like(xd), torch.zeros_like(od), torch.zeros_like(wd)
    _C.deform_conv_backward_input(xd, od, gd, gi, goff, wd, bufs[0], wd.size(3), wd.size(2), 1, 1, 1, 1, 1, 1, grp, 1, 2)
    _C.deform_conv_backward_filter(xd, od, gd, gw, bufs[0], bufs[1], wd.size(3), wd.size(2), 1, 1, 1, 1, 1, 1, grp, 1, 1, 2)
    r = orc.deform_conv_backward(x, off, None, wt, go, 1, 1, 1, grp, 1, False)
    close(gi, r[0], "gx"), close(goff, r[1], "goff"), close(gw, r[3], "gw")
    # ---- DCNv2: forward (:205-242), backward (:244-295)
    out = xd.new_empty(n, co, h, w)
    _C.modulated_deform_conv_forward(xd, wd, bd, bufs[0], od, md, out, bufs[1], 3, 3, 1, 1, 1, 1, 1, 1, grp, 1, True)
    close(out, orc.deform_conv_forward(x, off, mask, wt, bias, 1, 1, 1, grp, 1), "y2")
    gi, goff, gm = torch.zeros_like(xd), torch.zeros_like(od), torch.zeros_like(md)
    gw, gb = torch.zeros_like(wd), torch.zeros_like(bd)
    _C.modulated_deform_conv_backward(xd, wd, bd, bufs[0], od, md, bufs[1], gi, gw, gb, goff, gm, gd, 3, 3, 1, 1, 1, 1, 1, 1,
                                      grp, 1, True)
    r = orc.deform_conv_backward(x, off, mask, wt, go, 1, 1, 1, grp, 1, True)
    for a, b, nm in zip((gi, goff, gm, gw, gb), r, ("gx", "goff", "gmask", "gw", "gb")):
        close(a, b, nm)
