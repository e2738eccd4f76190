"""ctypes binding of include/rainbow_b200.h.

The product path has NO CPU fallback: if librainbow_b200.so is missing and cannot be built, or a
kernel is asked to run on a non-CUDA tensor, this module raises.
"""
import ctypes as C
import os

from . import _build

_lib = None

_vp, _i64, _i32, _f32, _u64 = C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_uint64

class HeadParams(C.Structure):
    """rb_head_params of include/rainbow_b200.h (device pointers of one net's noisy dueling head)."""
    _fields_ = [(n, _vp * 2) for n in ("w1_mu", "w1_sigma", "b1_mu", "b1_sigma", "w2_mu", "w2_sigma", "b2_mu", "b2_sigma",
                                        "eps_in1", "eps_out1", "eps_in2", "eps_out2")] + \
               [(n, C.c_int) for n in ("conv_features", "hidden", "atoms", "actions")]


class HeadGrads(C.Structure):
    """rb_head_grads: where rb_head_backward writes the 16 parameter gradients."""
    _fields_ = [(n, _vp * 2) for n in ("w1_mu", "w1_sigma", "b1_mu", "b1_sigma", "w2_mu", "w2_sigma", "b2_mu", "b2_sigma")]


_hp, _hg = C.POINTER(HeadParams), C.POINTER(HeadGrads)

# name -> (restype, argtypes); must list every symbol declared in include/rainbow_b200.h
SIGNATURES = {
    "rb_abi_version": (C.c_int, []),
    "rb_last_error": (C.c_char_p, []),
    "rb_profile_enable": (C.c_int, [_i32]),
    "rb_profile_collect": (C.c_int, [_i32, C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "rb_tree_update": (C.c_int, [_vp, _i64, _i64, _vp, _vp, _f32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "rb_tree_find": (C.c_int, [_vp, _i64, _i64, _vp, _i32, _vp, _vp, _vp, _vp]),
    "rb_tree_sample": (C.c_int, [_vp, _i64, _i64, _vp, _i32, _i32, _vp, _i32, _u64, _vp, _i32, _f32, _vp, _i32,
                                 _vp, _vp, _vp, _vp, _vp, _vp]),
    "rb_gather": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rb_iter_states": (C.c_int, [_vp, _vp, _i64, _i64, _i32, _i32, _vp, _vp]),
    "rb_append": (C.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int32, _f32, _i32, _vp]),
    "rb_append_batch": (C.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp]),
    "rb_c51_loss_grad": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _f32, _f32, _i32, _i32, _i32,
                                   _vp, _vp, _vp, _vp, _vp]),
    "rb_noisy_resample": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _u64, _vp, _vp]),
    "rb_noisy_outer": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "rb_noise_factors": (C.c_int, [_vp, _i32, _vp, _i32, _vp, _vp, _u64, _vp, _vp]),
    "rb_head_splits": (C.c_int, [_i32, _i32, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "rb_head_ticket_count": (C.c_int, []),
    "rb_head_supported": (C.c_int, [_i32, _i32, _i32, _i32, _i32, _i32]),
    "rb_head_debug": (C.c_int, [_i32]),
    "rb_head_forward": (C.c_int, [_hp, _vp, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rb_head_logits": (C.c_int, [_vp, _i32, _i32, _i32, _vp, _vp]),
    "rb_head_backward": (C.c_int, [_hp, _hg, _vp, _vp, _vp, _i32, _vp, _vp, _i32, _i32, _vp]),
    "rb_bias_grad": (C.c_int, [_vp, _i32, _i32, _i32, _vp, _vp]),
    "rb_conv_wgrad_scratch_elems": (C.c_int, [_i32, _i32, _i32, _i32, _i32, _i32]),
    "rb_conv_wgrad": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "rb_conv_forward": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "rb_c51_dueling_loss_grad": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _f32, _f32, _i32,
                                           _vp, _vp, _vp, _vp, _vp]),
    "rb_noisy_compose": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "rb_peer_scratch_bytes": (C.c_int, []),
    "rb_peer_reduce": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i64, _i64, _f32, _vp, _vp, _vp, _vp]),
    "rb_peer_adam_gather": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _f32, _f32, _f32,
                                      _vp, _vp, _vp, _vp, _vp, _vp]),
    "rb_peer_clip_adam": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i64, _vp, _vp, _vp, _f32, _f32, _f32, _f32, _f32, _f32,
                                    _vp, _vp, _vp, _vp, _vp]),
    "rb_clip_adam_scratch_elems": (C.c_int, []),
    "rb_clip_adam": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _f32, _f32, _vp, _vp, _vp, _vp, _vp]),
    "rb_q_values": (C.c_int, [_vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
}


class RainbowB200Error(RuntimeError):
    pass


def load():
    """Load (building first if the .so is absent or older than its source) and type the C ABI."""
    global _lib
    if _lib is not None:
        return _lib
    if _build.stale():
        try:
            _build.build()
        except Exception as e:  # no silent fallback
            if not os.path.exists(_build.SO):
                raise RainbowB200Error(f"librainbow_b200.so is missing and could not be built: {e}") from e
    lib = C.CDLL(_build.SO)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.rb_abi_version() != 2:
        raise RainbowB200Error("librainbow_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RainbowB200Error(f"rainbow_b200 C ABI error {rc}: {load().rb_last_error().decode()}")


def ptr(t):
    """Device pointer of a CUDA tensor (None -> NULL).  Refuses host tensors: there is no CPU path."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RainbowB200Error("rainbow_b200 kernels need CUDA tensors (no CPU fallback exists)")
    if not t.is_contiguous():
        raise RainbowB200Error("rainbow_b200 kernels need contiguous tensors")
    return t.data_ptr()


def stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


KERNEL_IDS = ["tree_update", "tree_find", "tree_sample", "gather", "iter_states", "append", "c51", "noisy_resample",
              "noisy_compose", "sqnorm", "clip_adam", "head_fc1", "head_fc2", "head_logits", "head_wgrad2", "head_dh",
              "head_bwd1", "noise_factors", "c51_dueling", "bias_grad", "q_values", "head_reduce1", "conv_wgrad", "conv_fwd"]  # order of the enum in include/rainbow_b200.h


class KernelTimer:
    """with KernelTimer() as kt: ...eager (non-graph) work... ; kt.result -> {kernel: (launches, mean_us)}"""

    def __enter__(self):
        check(load().rb_profile_enable(1))
        return self

    def __exit__(self, *exc):
        lib = load()
        check(lib.rb_profile_enable(0))
        self.result = {}
        for i, name in enumerate(KERNEL_IDS):
            ms, n = C.c_double(0.0), C.c_int(0)
            check(lib.rb_profile_collect(i, C.byref(ms), C.byref(n)))
            if n.value:
                self.result[name] = (n.value, 1e3 * ms.value / n.value)
        return False
