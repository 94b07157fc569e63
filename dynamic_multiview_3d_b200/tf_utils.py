"""Operator-level drop-in surface: the reference's op helpers, same names and argument
meaning (dyn_mult_view/mv3d/utils/tf_utils.py:18-98), backed by libdmv3d.so.

Differences forced by the host framework (PyTorch tensors instead of a TF graph):
  * tensors are NHWC ``torch.Tensor`` on a CUDA device -- bf16 activations, fp32 images,
    flows and losses; variables live in the active ``VariableStore`` (variables.py) under
    the reference's names ``name/w``, ``name/b``, ``name/Matrix``;
  * ``conv2d_msra`` / ``deconv2d_msra`` / ``linear_msra`` take an optional ``act=`` so the
    activation is fused into the kernel epilogue; ``lrelu(conv2d_msra(...))`` composes too.
"""
import math

import torch

from . import functional as F
from .variables import current_store


def _rec(store, var, y):
    """Test hooks: ``store.record`` (dict) receives every layer's output under the layer's name; ``store.record_grad``
    (dict) the gradient that output receives in backward -- (kind, tensor) with kind "pre" when the consuming layer's
    dgrad already applied the activation derivative (functional.py: activation-derivative fusion; the tensor is then the
    gradient w.r.t. the layer's PRE-activation), else "out"."""
    if store.record is not None:
        name = var.name.rsplit("/", 1)[0]
        store.record[name] = y
        rg = getattr(store, "record_grad", None)
        if rg is not None and y.requires_grad:
            cell = getattr(y, "_dmv_cell", None)
            y.register_hook(lambda g, name=name, cell=cell: rg.__setitem__(name, ("pre" if (cell is not None and cell.fused) else "out", g.detach())))
    return y


def euclidean_loss(input1, input2):
    """tf_utils.py:18-19  reduce_mean(reduce_sum((a-b)^2, 3))."""
    return F.reconstruction_loss(input1, input2, "l2")


def l1_loss(input1, input2):
    """tf_utils.py:22-23  reduce_mean(reduce_sum(|a-b|, 3))."""
    return F.reconstruction_loss(input1, input2, "l1")


def relu(x, name="relu"):
    """tf_utils.py:25-27  0.5x + 0.5|x|."""
    return F.activation(x, "relu")


def lrelu(x, leak=0.2, name="lrelu"):
    """tf_utils.py:29-33  f1 x + f2 |x|; the kernels implement the reference's leak 0.2."""
    if leak != 0.2:
        raise ValueError("only the reference's leak=0.2 is implemented")
    return F.activation(x, "lrelu")


def coords(h, w, batch_size, device="cuda"):
    """tf_utils.py:44-52: [B,h,w,2] with channel 0 = ROW index (Y), channel 1 = COLUMN index (X).
    Inspection helper only -- the training path forms the grid inside the sampler kernel."""
    y = torch.arange(h, dtype=torch.float32, device=device)
    x = torch.arange(w, dtype=torch.float32, device=device)
    Y, X = torch.meshgrid(y, x, indexing="ij")
    return torch.stack((Y, X), dim=2).unsqueeze(0).repeat(batch_size, 1, 1, 1)


def warp_pts_layer(flow_field, name="warp_pts"):
    """tf_utils.py:35-38  flow + coords.  Inspection helper (see coords)."""
    b, h, w, _ = flow_field.shape
    return flow_field + coords(h, w, b, flow_field.device)


def resample_layer(src_img, warp_pts, name="tgt_img"):
    """tf_utils.py:40-42  tf.contrib.resampler.resampler(src_img, warp_pts)."""
    return F.resampler(src_img, warp_pts)


def flow_resample_layer(src_img, flow_field, grid_order="ref_yx", name="tgt_img"):
    """resample_layer(src, warp_pts_layer(flow)) in one kernel (grid never materialised).
    grid_order 'ref_yx' reproduces the reference's (Y,X) grid; 'xy' is the un-transposed one."""
    return F.flow_resampler(src_img, flow_field, grid_order)


def linear_msra(input_, output_size, name, act=None, algo=None, group=1):
    """tf_utils.py:54-67: x @ Matrix[K,N] + b, Matrix ~ N(0, sqrt(2/K)), b = 0.  group > 1: each output row is repeated
    ``group`` times (functional.linear)."""
    store = current_store()
    fan_in = int(input_.shape[-1])
    with store.scope(name):
        matrix = store.get("Matrix", [fan_in, output_size], "normal", math.sqrt(2.0 / float(fan_in)))
        b = store.get("b", [output_size], "zeros")
    return _rec(store, matrix, F.linear(input_, matrix, b, act, algo, group))


def conv2d_msra(input_, output_dim, k_h, k_w, d_h, d_w, name, act=None, algo=None, out_dtype=torch.bfloat16):
    """tf_utils.py:70-84: conv2d(x, w[kh,kw,Cin,Cout], SAME) + b, w ~ truncated N(0, sqrt(2/(kh kw Cin)))."""
    if d_h != d_w:
        raise ValueError("only equal strides are implemented (all reference layers use them)")
    store = current_store()
    cin = int(input_.shape[-1])
    with store.scope(name):
        w = store.get("w", [k_h, k_w, cin, output_dim], "truncated_normal", math.sqrt(2.0 / float(k_h * k_w * cin)))
        b = store.get("b", [output_dim], "zeros")
    return _rec(store, w, F.conv2d(input_, w, b, d_h, act, algo, out_dtype))


def deconv2d_msra(input_, output_shape, k_h, k_w, d_h, d_w, name, act=None, algo=None, out_dtype=torch.bfloat16):
    """tf_utils.py:87-98: conv2d_transpose(x, w[kh,kw,Cout,Cin], output_shape, strides) (SAME, no bias),
    w ~ N(0, sqrt(2/(kh kw Cin) * dh * dw))."""
    if d_h != d_w:
        raise ValueError("only equal strides are implemented (all reference layers use them)")
    store = current_store()
    cin = int(input_.shape[-1])
    with store.scope(name):
        w = store.get("w", [k_h, k_w, int(output_shape[-1]), cin], "normal",
                      math.sqrt(2.0 / float(k_h * k_w * cin) * float(d_h) * float(d_w)))
    return _rec(store, w, F.deconv2d(input_, w, (output_shape[1], output_shape[2]), d_h, act, algo, out_dtype))
