"""ctypes binding of libdmv3d.so (include/dmv3d.h).

The library is the product: if it is missing or a call fails, this module raises --
there is no CPU or PyTorch fallback anywhere on the path.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdmv3d.so")

OK = 0
ACT = {None: 0, "none": 0, "lrelu": 1, "relu": 2, "tanh": 3}
LOSS = {"l2": 0, "l1": 1}
DT_BF16, DT_F32, DT_S2D = 0, 1, 2
ALGO = {"auto": 0, "simt": 1, "tcgen05": 2}
ALGO_PACK_ONLY, ALGO_PREPACKED = 0x100, 0x200
SAMPLER_ADD_GRID, SAMPLER_GRID_XY = 1, 2

_vp, _i, _ll, _f, _sz, _u = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_size_t, C.c_uint

# name -> (restype, argtypes); every name here must be declared in include/dmv3d.h
SIGNATURES = {
    "dmv_version": (_i, []),
    "dmv_arch": (C.c_char_p, []),
    "dmv_last_error": (_i, [C.c_char_p, _sz]),
    "dmv_launch_count": (_ll, []),
    "dmv_tc_launch_count": (_ll, []),
    "dmv_launch_count_named": (_ll, [C.c_char_p]),
    "dmv_sampler_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _u, _vp]),
    "dmv_sampler_fwd_shared_src": (_i, [_vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _u, _vp]),
    "dmv_sampler_bwd_workspace_size": (_sz, [_i, _i, _i, _i, _i, _i]),
    "dmv_sampler_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _u, _vp, _sz, _vp]),
    "dmv_sampler_loss_workspace_size": (_sz, [_i, _i, _i]),
    "dmv_sampler_loss_fused": (_i, [_vp, _vp, _vp, C.POINTER(_f), _i, _f, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _u, _vp, _sz, _vp]),
    "dmv_sampler_loss_fused_shared_src": (_i, [_vp, _i, _i, _vp, _vp, C.POINTER(_f), _i, _f, _vp, _vp, _vp, _i, _i, _i, _i, _i, _u, _vp, _sz, _vp]),
    "dmv_sampler_grad_flow_shared_src": (_i, [_vp, _i, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _u, _vp]),
    "dmv_sampler_fuse_views_loss": (_i, [_vp, _i, _vp, _vp, C.POINTER(_f), _i, _f, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _u, _vp, _sz,
                                         _vp]),
    "dmv_loss_workspace_size": (_sz, [_ll]),
    "dmv_loss_fused_fwd_bwd": (_i, [_vp, _vp, _i, _vp, _vp, C.POINTER(_f), _i, _f, _vp, _vp, _vp, _vp, _ll, _i, _vp, _sz, _vp]),
    "dmv_scale_by_device_scalar": (_i, [_vp, _vp, _ll, _vp]),
    "dmv_conv_workspace_size": (_sz, [_i] * 8),
    "dmv_u8_to_f32": (_i, [_vp, _vp, _ll, _f, _vp]),
    "dmv_u8_crop_resize_bicubic": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _f, _vp]),
    "dmv_thin_s2d_size": (_sz, [_i] * 8),
    "dmv_thin_s2d_prep": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _vp]),
    "dmv_conv2d_fwd": (_i, [_vp, _i, _vp, _vp, _vp, _i] + [_i] * 9 + [_vp, _sz, _i, _vp]),
    "dmv_conv2d_dgrad": (_i, [_vp, _vp, _vp, _vp, _i] + [_i] * 8 + [_vp, _sz, _i, _vp]),
    "dmv_wgrad_workspace_size": (_sz, [_i] * 8),
    "dmv_conv2d_wgrad": (_i, [_vp, _i, _vp, _vp, _vp] + [_i] * 8 + [_vp, _sz, _i, _vp]),
    "dmv_deconv2d_fwd": (_i, [_vp, _vp, _vp, _i] + [_i] * 9 + [_vp, _sz, _i, _vp]),
    "dmv_deconv2d_dgrad": (_i, [_vp, _i, _vp, _vp, _vp, _i] + [_i] * 8 + [_vp, _sz, _i, _vp]),
    "dmv_deconv2d_wgrad": (_i, [_vp, _vp, _i, _vp] + [_i] * 8 + [_vp, _sz, _i, _vp]),
    "dmv_linear_fwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _sz, _i, _vp]),
    "dmv_linear_dgrad": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _sz, _i, _vp]),
    "dmv_linear_wgrad": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _sz, _i, _vp]),
    "dmv_act_fwd": (_i, [_vp, _vp, _i, _ll, _i, _vp]),
    "dmv_act_bwd": (_i, [_vp, _vp, _vp, _i, _ll, _i, _vp]),
    "dmv_act_bwd_bias_workspace_size": (_sz, [_ll, _i]),
    "dmv_act_bwd_bias": (_i, [_vp, _vp, _vp, _vp, _ll, _i, _i, _vp, _sz, _vp]),
    "dmv_act_bwd_bias_grouped": (_i, [_vp, _ll, _i, _vp, _vp, _vp, _ll, _i, _i, _vp, _sz, _vp]),
    "dmv_cast_f32_to_bf16": (_i, [_vp, _vp, _ll, _vp]),
    "dmv_cast_bf16_to_f32": (_i, [_vp, _vp, _ll, _vp]),
    "dmv_adam_tick": (_i, [_vp, _f, _f, _f, _vp]),
    "dmv_adam_multi": (_i, [C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp),
                            C.POINTER(_ll), _i, _vp, _f, _f, _f, _f, _vp]),
    "dmv_adam_multi_gated": (_i, [C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp),
                                  C.POINTER(_ll), _i, _vp, _f, _f, _f, _f, _vp, _vp]),
    "dmv_set_flag": (_i, [_vp, _i, _vp]),
    "dmv_linear_wgrad_adam": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _f, _f, _f, _f, _vp]),
    "dmv_dp_signal_words": (_i, [_i]),
    "dmv_dp_exchange_chunk": (_i, [C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), _vp, _vp, _vp, _vp, _vp, _vp, _ll, _ll,
                                   _i, _i, _i, _i, _vp, _f, _f, _f, _f, _i, _vp]),
}

_lib = None


class DmvError(RuntimeError):
    pass


def load():
    """Load libdmv3d.so (built in-tree by ``__graft_entry__.build()`` / csrc/Makefile)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DmvError(
                "libdmv3d.so not found at %s -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C dynamic_multiview_3d_b200/csrc`; there is no fallback path." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error():
    buf = C.create_string_buffer(512)
    load().dmv_last_error(buf, 512)
    return buf.value.decode("utf-8", "replace")


def check(rc, what=""):
    if rc != OK:
        raise DmvError("%s failed (code %d): %s" % (what or "libdmv3d call", rc, last_error()))


def call(name, *args):
    check(getattr(load(), name)(*args), name)


def launch_count():
    return int(load().dmv_launch_count())


def tc_launch_count():
    return int(load().dmv_tc_launch_count())


def launch_count_named(what):
    """Launches so far of the kernel form labelled ``what`` (the label of its launch check in csrc/)."""
    return int(load().dmv_launch_count_named(what.encode()))
