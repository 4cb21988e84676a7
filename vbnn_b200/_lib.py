"""ctypes binding of libvbnn.so (include/vbnn.h).  No CPU fallback: if the shared library is
missing this module raises, and every compute entry point fails with VBNN_E_CUDA when there is
no B200 to run on."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvbnn.so")

VBNN_OK = 0
E_INVALID, E_CUDA, E_NOMEM, E_UNSUPPORTED, E_NCCL, E_STATE = -1, -2, -3, -4, -5, -6
REPARAM_WEIGHT, REPARAM_LOCAL = 0, 1
PREC_FP32, PREC_BF16 = 0, 1
KIND_VB, KIND_LINEAR = 0, 1
(BUF_MEANS, BUF_LVARS, BUF_BIAS, BUF_WEIGHT, BUF_GRAD_WEIGHT, BUF_GRAD_SUM, BUF_GRAD_BIAS,
 BUF_ADAM_M_MU, BUF_ADAM_V_MU, BUF_ADAM_M_VAR, BUF_ADAM_V_VAR, BUF_EPS, BUF_STDV,
 BUF_MU_SQE, BUF_PRIOR_MEANS, BUF_PRIOR_LVARS) = range(16)
PRIOR_EMPIRICAL, PRIOR_FIXED, PRIOR_PER_WEIGHT = 0, 1, 2
PRIOR_KINDS = {"empirical": PRIOR_EMPIRICAL, "fixed": PRIOR_FIXED, "per_weight": PRIOR_PER_WEIGHT}
OUTPUT_RAW, OUTPUT_GAUSSIAN = 0, 1
OUTPUT_MODELS = {"raw": OUTPUT_RAW, "gaussian": OUTPUT_GAUSSIAN}


class VbnnOpts(C.Structure):
    _fields_ = [("var_init", C.c_float), ("msr_init", C.c_int), ("mu_init", C.c_float),
                ("B", C.c_float), ("S", C.c_int), ("lr_bias", C.c_float), ("lr_mu", C.c_float),
                ("lr_var", C.c_float), ("adam_beta1", C.c_float), ("adam_beta2", C.c_float),
                ("adam_eps", C.c_float), ("reparam", C.c_int), ("precision", C.c_int),
                ("strict_reference", C.c_int)]


# the fields vbnn_layer_set_opts may change (the reference reads them at every update), in the order
# MLP.state_dict() stores them
LIVE_OPTS = ("B", "lr_bias", "lr_mu", "lr_var", "adam_beta1", "adam_beta2", "adam_eps")


class VbnnStats(C.Structure):
    _fields_ = [(n, C.c_float) for n in (
        "vlc_grad", "vle_grad", "mlc_grad", "mle_grad", "min_variance", "max_variance",
        "mean_variance", "var_hat", "mean_means", "std_means", "min_means", "max_means",
        "mu_normratio", "var_normratio")]


# the reference's Log ids (VBLinear.lua:150-163), in struct order
STAT_NAMES = ["vlc grad", "vle grad", "mlc grad", "mle grad", "min variance", "max variance",
              "mean variance", "var hat", "mean means", "std means", "min. means", "max. means",
              "mu normratio", "var normratio"]

_P = C.c_void_p
_F = C.POINTER(C.c_float)
_PROTOS = {
    "vbnn_abi_version": (C.c_int, []),
    "vbnn_last_error": (C.c_char_p, []),
    "vbnn_opts_default": (None, [C.POINTER(VbnnOpts)]),
    "vbnn_ctx_create": (C.c_int, [C.c_int, _P, C.c_uint64, C.POINTER(_P)]),
    "vbnn_ctx_create_ex": (C.c_int, [C.c_int, _P, C.c_int, C.c_uint64, C.POINTER(_P)]),
    "vbnn_ctx_destroy": (C.c_int, [_P]),
    "vbnn_ctx_synchronize": (C.c_int, [_P]),
    "vbnn_ctx_profile": (C.c_int, [_P, C.c_int]),
    "vbnn_ctx_profile_read": (C.c_int, [_P, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.POINTER(C.c_double)]),
    "vbnn_ctx_phase_read": (C.c_int, [_P, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    "vbnn_ctx_set_step": (C.c_int, [_P, C.c_uint32]),
    "vbnn_ctx_get_step": (C.c_int, [_P, C.POINTER(C.c_uint32)]),
    "vbnn_layer_create": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.POINTER(VbnnOpts), C.POINTER(_P)]),
    "vbnn_layer_destroy": (C.c_int, [_P]),
    "vbnn_layer_dims": (C.c_int, [_P, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vbnn_layer_sample": (C.c_int, [_P, C.c_int, _P]),
    "vbnn_layer_clamp_to_map": (C.c_int, [_P]),
    "vbnn_layer_forward": (C.c_int, [_P, _P, C.c_int, _P, _P]),
    "vbnn_layer_backward_data": (C.c_int, [_P, _P, _P, C.c_int, _P]),
    "vbnn_layer_acc_grad": (C.c_int, [_P, _P, _P, C.c_int, C.c_float]),
    "vbnn_layer_reset_acc": (C.c_int, [_P]),
    "vbnn_layer_compute_prior": (C.c_int, [_P, _F, _F]),
    "vbnn_layer_grads": (C.c_int, [_P, _P, _P, _P, _P]),
    "vbnn_layer_update": (C.c_int, [_P, C.POINTER(VbnnStats)]),
    "vbnn_layer_calc_lc": (C.c_int, [_P, _P, _F]),
    "vbnn_layer_set_prior": (C.c_int, [_P, C.c_int, C.c_float, C.c_float]),
    "vbnn_layer_get_prior": (C.c_int, [_P, C.POINTER(C.c_int), _F, _F]),
    "vbnn_layer_get_opts": (C.c_int, [_P, C.POINTER(VbnnOpts)]),
    "vbnn_layer_set_opts": (C.c_int, [_P, C.POINTER(VbnnOpts)]),
    "vbnn_mlp_set_opts": (C.c_int, [_P, C.POINTER(VbnnOpts)]),
    "vbnn_layer_get": (C.c_int, [_P, C.c_int, _P]),
    "vbnn_layer_set": (C.c_int, [_P, C.c_int, _P]),
    "vbnn_layer_device_ptr": (C.c_int, [_P, C.c_int, C.POINTER(_P), C.POINTER(C.c_size_t)]),
    "vbnn_layer_bind": (C.c_int, [_P, C.c_int, _P]),
    "vbnn_layer_get_t": (C.c_int, [_P, C.POINTER(C.c_int)]),
    "vbnn_layer_set_t": (C.c_int, [_P, C.c_int]),
    "vbnn_layer_snr_count": (C.c_int, [_P, C.c_float, _P, C.POINTER(C.c_longlong)]),
    "vbnn_layer_draw_noise": (C.c_int, [_P, C.c_uint32, C.c_int, C.c_int, C.c_int, _P]),
    "vbnn_mlp_create": (C.c_int, [_P, C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, C.POINTER(VbnnOpts), C.POINTER(_P)]),
    "vbnn_mlp_destroy": (C.c_int, [_P]),
    "vbnn_mlp_num_layers": (C.c_int, [_P]),
    "vbnn_mlp_layer": (C.c_int, [_P, C.c_int, C.POINTER(_P)]),
    "vbnn_mlp_init_params": (C.c_int, [_P, C.c_uint64, C.c_int]),
    "vbnn_mlp_reset_gradients": (C.c_int, [_P]),
    "vbnn_mlp_sample": (C.c_int, [_P, C.c_int]),
    "vbnn_mlp_run": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, _F, _F]),
    "vbnn_mlp_update": (C.c_int, [_P]),
    "vbnn_mlp_calc_lc": (C.c_int, [_P, _F]),
    "vbnn_mlp_step": (C.c_int, [_P, _P, _P, C.c_int, _P]),
    "vbnn_mlp_step_grad_input": (C.c_int, [_P, _P, _P, C.c_int, _P, _P]),
    "vbnn_mlp_forward_train": (C.c_int, [_P, _P, C.c_int, _P]),
    "vbnn_mlp_backward_update": (C.c_int, [_P, _P, _P]),
    "vbnn_mlp_step_host": (C.c_int, [_P, _P, _P, C.c_int, _F, _F]),
    "vbnn_mlp_submit_host": (C.c_int, [_P, _P, _P, C.c_int]),
    "vbnn_mlp_collect": (C.c_int, [_P, _F, _F]),
    "vbnn_mlp_submit_host_u8": (C.c_int, [_P, _P, _P, C.c_int, C.c_float, C.c_float]),
    "vbnn_mlp_join_streams": (C.c_int, [_P]),
    "vbnn_mlp_test": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, _F, _F]),
    "vbnn_mlp_predict": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P, _P, _F, _F]),
    "vbnn_mlp_predict_outputs": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _F, _F]),
    "vbnn_mlp_get_outputs": (C.c_int, [_P, C.c_int, _P]),
    "vbnn_mlp_launch_count": (C.c_int, [_P, C.POINTER(C.c_longlong)]),
    "vbnn_mlp_graph_captures": (C.c_int, [_P, C.POINTER(C.c_longlong)]),
    "vbnn_mlp_grad_arena": (C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_size_t)]),
    "vbnn_comm_unique_id": (C.c_int, [_P]),
    "vbnn_comm_init": (C.c_int, [_P, _P, C.c_int, C.c_int]),
    "vbnn_comm_destroy": (C.c_int, [_P]),
    "vbnn_comm_allreduce": (C.c_int, [_P, _P, C.c_size_t]),
    "vbnn_mlp_peer_export": (C.c_int, [_P, _P, C.c_size_t, C.POINTER(C.c_size_t)]),
    "vbnn_mlp_peer_import": (C.c_int, [_P, _P, C.c_size_t]),
    "vbnn_mlp_peer_active": (C.c_int, [_P]),
    "vbnn_mlp_sync_replicas": (C.c_int, [_P]),
    "vbnn_peer_shard": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vbnn_gemm_bf16": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, C.c_int, C.c_int, _P, C.c_int,
                                 C.c_int, C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_longlong,
                                 C.c_longlong]),
    "vbnn_philox_normal": (C.c_int, [_P, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int,
                                     C.c_int, C.c_int, _P]),
    "vbnn_debug_knob": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(C.c_int)]),
}

STREAM_GIVEN, STREAM_LEGACY_DEFAULT, STREAM_PRIVATE_BLOCKING = 0, 1, 2
KNOB_DEFAULT = -2 ** 31

_lib = None


class VbnnError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libvbnn error {code}: {msg}")
        self.code = code


def lib():
    """Load libvbnn.so (once).  Raises ImportError if it has not been built: there is no
    fallback implementation."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a).  vbnn_b200 has no CPU or PyTorch fallback.")
    l = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(l, name)
        fn.restype = res
        fn.argtypes = args
    _lib = l
    return l


def check(code):
    if code != VBNN_OK:
        raise VbnnError(code, lib().vbnn_last_error().decode("utf-8", "replace"))
    return code


def knob(name, value=KNOB_DEFAULT):
    """Set an experiment switch of libvbnn.so (csrc/knobs.h); returns the previous value.
    knob(name) restores the default / environment value."""
    old = C.c_int()
    check(lib().vbnn_debug_knob(name.encode(), int(value), C.byref(old)))
    return old.value
