"""ctypes binding of libb200gan.so (the C ABI declared in include/b200gan.h).

The product path has no CPU or cuDNN fallback: if the shared library is missing, or an entry point
returns an error, a RuntimeError is raised.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200gan.so")

c_i32, c_i64, c_f32, c_f64 = ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_double
c_vp, c_sz = ctypes.c_void_p, ctypes.c_size_t

ACT_NONE, ACT_LRELU, ACT_RELU, ACT_TANH, ACT_SIGMOID = 0, 1, 2, 3, 4
ALGO_AUTO, ALGO_SIMT, ALGO_TC = 0, 1, 2
PAD_ZERO, PAD_REFLECT = 0, 1
PACK_SIMT_FPROP, PACK_SIMT_DGRAD, PACK_TC_FPROP, PACK_TC_DGRAD, PACK_TC_FPROP_UP2, PACK_TC_DGRAD_UP2 = range(6)


class ConvGeom(ctypes.Structure):
    _fields_ = [(n, c_i32) for n in (
        "N", "H", "W", "C", "K", "R", "S", "stride", "pad_t", "pad_l", "pad_b", "pad_r",
        "pad_mode", "up", "transposed", "P", "Q")]

    def key(self):
        return tuple(getattr(self, n) for n, _ in self._fields_)


class Epilogue(ctypes.Structure):
    _fields_ = [("bias", c_vp), ("act", c_i32), ("slope", c_f32), ("chan_scale", c_vp),
                ("stats", c_vp), ("stats_per_sample", c_i32), ("round_tf32", c_i32)]


class NormDesc(ctypes.Structure):
    _fields_ = [("N", c_i32), ("HW", c_i32), ("C", c_i32), ("per_sample", c_i32), ("eps", c_f32),
                ("momentum", c_f32), ("act", c_i32), ("slope", c_f32), ("round_tf32", c_i32)]


class GpMlpDesc(ctypes.Structure):
    _fields_ = [("N", c_i32), ("Din", c_i32), ("H1", c_i32), ("H2", c_i32), ("slope", c_f32),
                ("lambda_gp", c_f32)]


class PackJob(ctypes.Structure):
    _fields_ = [("w", c_vp), ("packed", c_vp), ("geom", ConvGeom), ("pack", c_i32)]


class NbBn(ctypes.Structure):
    _fields_ = [("stats", c_vp), ("gamma", c_vp), ("beta", c_vp), ("eps", c_f32), ("count", c_f64), ("groups", c_i32),
                ("reserved", c_i32)]


class TailDesc(ctypes.Structure):
    _fields_ = [("N", c_i32), ("H", c_i32), ("W", c_i32), ("C", c_i32), ("K", c_i32), ("act_mid", c_i32),
                ("slope", c_f32), ("act_out", c_i32)]


class AdamTensor(ctypes.Structure):
    _fields_ = [("p", c_vp), ("g", c_vp), ("m", c_vp), ("v", c_vp), ("n", c_i64)]


# name -> (restype, argtypes); must list every function declared in include/b200gan.h
_P = ctypes.POINTER
SIGNATURES = {
    "b200gan_version": (c_i32, []),
    "b200gan_last_error": (ctypes.c_char_p, []),
    "b200gan_check_device": (c_i32, []),
    "b200gan_packed_weight_floats": (c_sz, [_P(ConvGeom), c_i32]),
    "b200gan_pack_weights": (c_i32, [_P(ConvGeom), c_i32, c_vp, c_vp, c_vp]),
    "b200gan_pack_weights_multi": (c_i32, [_P(PackJob), c_i32, c_vp]),
    "b200gan_conv2d_supported": (c_i32, [_P(ConvGeom), c_i32, c_i32]),
    "b200gan_conv2d_fprop": (c_i32, [_P(ConvGeom), _P(Epilogue), c_vp, c_vp, c_vp, c_i32, c_vp]),
    "b200gan_conv2d_dgrad_workspace_floats": (c_sz, [_P(ConvGeom), c_i32]),
    "b200gan_conv2d_dgrad": (c_i32, [_P(ConvGeom), c_vp, c_vp, c_vp, c_vp, c_i32, c_vp]),
    "b200gan_conv2d_wgrad_workspace_floats": (c_sz, [_P(ConvGeom), c_i32]),
    "b200gan_conv2d_wgrad": (c_i32, [_P(ConvGeom), c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp]),
    "b200gan_epilogue_bwd": (c_i32, [c_vp, c_vp, c_vp, c_i32, c_f32, c_i64, c_i32, c_i64, c_i32, c_vp, c_vp]),
    "b200gan_bias_grad": (c_i32, [c_vp, c_vp, c_vp, c_i32, c_f32, c_i64, c_i32, c_i64, c_vp, c_vp]),
    "b200gan_norm_stats": (c_i32, [_P(NormDesc), c_vp, c_vp, c_vp]),
    "b200gan_norm_finalize": (c_i32, [_P(NormDesc), c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "b200gan_norm_apply": (c_i32, [_P(NormDesc), c_vp, c_vp, c_vp, c_vp]),
    "b200gan_norm_bwd": (c_i32, [_P(NormDesc), c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "b200gan_norm_bwd_bwd": (c_i32, [_P(NormDesc)] + [c_vp] * 13),
    "b200gan_tail_supported": (c_i32, [_P(TailDesc)]),
    "b200gan_tail_fprop": (c_i32, [_P(TailDesc), c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "b200gan_tail_bwd_workspace_bytes": (c_sz, [_P(TailDesc)]),
    "b200gan_tail_bwd": (c_i32, [_P(TailDesc)] + [c_vp] * 10 + [c_i32, c_vp]),
    "b200gan_nchw_to_nhwc": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_vp]),
    "b200gan_nhwc_to_nchw": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_vp]),
    "b200gan_upsample2x_fwd": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp]),
    "b200gan_upsample2x_bwd": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp]),
    "b200gan_pad2d_fwd": (c_i32, [c_vp, c_vp] + [c_i32] * 10 + [c_vp]),
    "b200gan_pad2d_bwd": (c_i32, [c_vp, c_vp] + [c_i32] * 9 + [c_vp]),
    "b200gan_act_fwd": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_f32, c_i64, c_i32, c_i64, c_vp, c_vp]),
    "b200gan_gp_mlp_workspace_floats": (c_sz, [_P(GpMlpDesc)]),
    "b200gan_gp_mlp_fwd_bwd": (c_i32, [_P(GpMlpDesc)] + [c_vp] * 12),
    "b200gan_critic_step_workspace_floats": (c_sz, [_P(GpMlpDesc)]),
    "b200gan_critic_step_mlp": (c_i32, [_P(GpMlpDesc)] + [c_vp] * 18),
    "b200gan_adam_step": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_f64, c_f64, c_f64, c_f64, c_f32, c_vp, c_vp]),
    "b200gan_nb_supported": (c_i32, [_P(ConvGeom)]),
    "b200gan_nb_groups_supported": (c_i32, [_P(ConvGeom), c_i32]),
    "b200gan_nb_fprop": (c_i32, [_P(ConvGeom), _P(NbBn), c_vp, c_vp, c_vp, c_f32, c_vp, c_vp, c_vp, c_i32, c_f32, c_vp,
                                 c_vp, c_vp, c_i32, c_vp]),
    "b200gan_nb_dz": (c_i32, [c_i32, c_i64, c_i32, c_vp, c_vp, c_vp, c_i32, c_f32, _P(NbBn), c_vp, c_vp, c_vp, c_vp]),
    "b200gan_nb_wgrad_workspace_floats": (c_sz, [_P(ConvGeom)]),
    "b200gan_nb_wgrad": (c_i32, [_P(ConvGeom), _P(NbBn), c_vp, c_vp, c_vp, c_vp, c_vp]),
    "b200gan_nb_dgrad": (c_i32, [_P(ConvGeom), c_vp, c_vp, _P(NbBn), c_vp, c_vp, c_vp, c_vp]),
    "b200gan_nb_tail_fwd": (c_i32, [c_i32, c_i32, c_i32, _P(NbBn), c_vp, c_vp, c_vp, c_f32, c_vp, c_vp, c_i32, c_vp]),
    "b200gan_nb_tail_bwd": (c_i32, [c_i32, c_i32, c_i32, _P(NbBn), c_vp, c_vp, c_i32, c_vp, c_vp, c_vp]),
    "b200gan_linear1_fwd": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp]),
    "b200gan_linear1_bwd": (c_i32, [c_vp] * 7 + [c_i32, c_i32, c_i32, c_vp]),
    "b200gan_bce_fwd": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp]),
    "b200gan_bce_bwd": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "b200gan_adam_multi": (c_i32, [_P(AdamTensor), c_i32, c_f64, c_f64, c_f64, c_f64, c_f32, c_vp, c_vp]),
}

_lib = None


def load():
    """Load libb200gan.so (building it first when a toolchain and the sources are present)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: run `python pytorch-gan_b200/build.py` (or __graft_entry__.build()). "
            "b200gan has no CPU / cuDNN fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == the library does not export the ABI
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


CALLS = 0  # number of C-ABI launches issued by this process (each is >= 1 CUDA kernel)


def check(rc, what=""):
    global CALLS
    CALLS += 1
    if rc != 0:
        msg = load().b200gan_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libb200gan {what} failed (code {rc}): {msg}")
