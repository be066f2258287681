"""ctypes binding of libnint.so (include/nint.h).  No CPU fallback: a missing library or a
machine without a B200 makes every compute call raise."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NINT_LIB") or os.path.join(HERE, "libnint.so")   # NINT_LIB: A/B runs against another build
MAX_LAYERS = 8
DTYPE_BF16, DTYPE_TF32 = 0, 1
DTYPE_BYTES = {DTYPE_BF16: 2, DTYPE_TF32: 4}
X_FP32, X_BF16 = 0, 1
FLAG_DETERMINISTIC, FLAG_INPUT_GRAD, FLAG_STATE_GRAD, FLAG_TANGENT, FLAG_SECOND_ORDER = 1, 2, 4, 8, 16
FLAG_PARAM_TANGENT = 32
EXPORTS = ["nint_version", "nint_last_error", "nint_plan_create", "nint_plan_destroy", "nint_plan_workspace_bytes",
           "nint_plan_bind", "nint_plan_set_weights", "nint_plan_set_head", "nint_plan_reset_state",
           "nint_plan_set_state", "nint_plan_get_state", "nint_forward", "nint_forward_ex", "nint_forward_bank",
           "nint_plan_input_layout", "nint_pack_frames", "nint_backward", "nint_debug_raw_gates",
           "nint_gate_column", "nint_debug_read_trace", "nint_debug_fail_record", "nint_backward_bptt", "nint_backward_wgrad",
           "nint_backward_bptt_state", "nint_backward_initial_state", "nint_backward_input", "nint_backward_input_bank", "nint_forward_tangent",
           "nint_forward_tangent_bank", "nint_backward_second_order", "nint_backward_second_order_bank", "nint_plan_set_weight_tangent",
           "nint_plan_set_head_tangent", "nint_plan_clear_param_tangent", "nint_backward_second_order_params", "nint_cell_forward", "nint_cell_backward", "nint_loss_mse_l1",
           "nint_loss_mse_l1_bank", "nint_adam_step", "nint_adam_step_dev", "nint_dp_allreduce_adam", "nint_fuse_inputs", "nint_fuse_inputs_bank",
           "nint_fuse_inputs_adjoint", "nint_pick_tile", "nint_launch_count", "nint_plan_profile", "nint_plan_profile_read"]


class NintConfig(ctypes.Structure):
    _fields_ = [("batch", ctypes.c_int32), ("seq_len", ctypes.c_int32), ("height", ctypes.c_int32),
                ("width", ctypes.c_int32), ("in_channels", ctypes.c_int32), ("num_layers", ctypes.c_int32),
                ("hidden", ctypes.c_int32 * MAX_LAYERS), ("ksize", ctypes.c_int32 * MAX_LAYERS),
                ("dtype", ctypes.c_int32), ("training", ctypes.c_int32), ("return_sequence", ctypes.c_int32),
                ("flags", ctypes.c_int32)]


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -m nasa_niswan_b200.build` "
                           "(there is no CPU or PyTorch fallback for the ConvLSTM hot path)")
    L = ctypes.CDLL(LIB_PATH)
    vp, ci, fp = ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p  # device pointers travel as void*
    L.nint_version.restype = ci
    L.nint_last_error.restype = ctypes.c_char_p
    L.nint_plan_create.argtypes = [ctypes.POINTER(NintConfig), ctypes.POINTER(vp)]
    L.nint_plan_destroy.argtypes = [vp]
    L.nint_plan_destroy.restype = None
    L.nint_plan_workspace_bytes.argtypes = [vp]
    L.nint_plan_workspace_bytes.restype = ctypes.c_size_t
    L.nint_plan_bind.argtypes = [vp, vp, ctypes.c_size_t, vp]
    L.nint_plan_set_weights.argtypes = [vp, ci, fp, fp, vp]
    L.nint_plan_set_head.argtypes = [vp, fp, fp, vp]
    L.nint_plan_reset_state.argtypes = [vp, vp]
    L.nint_plan_set_state.argtypes = [vp, ci, fp, fp, vp]
    L.nint_plan_get_state.argtypes = [vp, ci, fp, fp, vp]
    L.nint_forward.argtypes = [vp, fp, fp, fp, vp]
    L.nint_forward_ex.argtypes = [vp, fp, ci, fp, fp, vp]
    L.nint_forward_bank.argtypes = [vp, fp, ctypes.c_longlong, fp, fp, fp, vp]
    L.nint_plan_input_layout.argtypes = [vp, ctypes.POINTER(ci), ctypes.POINTER(ci), ctypes.POINTER(ci)]
    L.nint_pack_frames.argtypes = [ci, fp, ci, ctypes.c_longlong, ci, ci, ci, ci, ci, fp, vp]
    L.nint_backward_input.argtypes = [vp, fp, vp]
    L.nint_backward_input_bank.argtypes = [vp, fp, vp]
    pp = ctypes.POINTER(vp)
    L.nint_forward_tangent.argtypes = [vp, fp, ci, pp, pp, fp, fp, pp, pp, vp]
    L.nint_forward_tangent_bank.argtypes = [vp, fp, ctypes.c_longlong, pp, pp, fp, fp, pp, pp, vp]
    L.nint_backward_second_order.argtypes = [vp, fp, fp, fp, fp, fp, fp, pp, pp, pp, pp, vp]
    L.nint_backward_second_order_bank.argtypes = [vp, fp, fp, fp, fp, fp, fp, pp, pp, pp, pp, vp]
    L.nint_plan_set_weight_tangent.argtypes = [vp, ci, fp, fp, vp]
    L.nint_plan_set_head_tangent.argtypes = [vp, fp, fp, vp]
    L.nint_plan_clear_param_tangent.argtypes = [vp, vp]
    L.nint_backward_second_order_params.argtypes = [vp, pp, pp, pp, pp, fp, fp, fp, fp, vp]
    L.nint_cell_forward.argtypes = [vp, fp, fp, fp, fp, fp, vp]
    L.nint_cell_backward.argtypes = [vp, fp, fp, fp, fp, fp, fp, fp, vp]
    L.nint_backward.argtypes = [vp, fp, fp, ctypes.POINTER(vp), ctypes.POINTER(vp), fp, fp, vp]
    L.nint_backward_bptt.argtypes = [vp, fp, fp, fp, fp, vp]
    L.nint_backward_wgrad.argtypes = [vp, ci, fp, fp, vp]
    L.nint_backward_bptt_state.argtypes = [vp, fp, fp, ctypes.POINTER(vp), ctypes.POINTER(vp), fp, fp, vp]
    L.nint_backward_initial_state.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(vp), vp]
    L.nint_debug_raw_gates.argtypes = [vp, fp, fp, vp]
    L.nint_launch_count.argtypes = [ci]
    L.nint_launch_count.restype = ctypes.c_longlong
    L.nint_plan_profile.argtypes = [vp, ci]
    L.nint_plan_profile_read.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_longlong)]
    L.nint_gate_column.argtypes = [ci, ci]
    L.nint_debug_read_trace.argtypes = [ctypes.POINTER(ctypes.c_longlong), ci, ci]
    L.nint_debug_fail_record.argtypes = [ctypes.POINTER(ctypes.c_ulonglong)]
    L.nint_loss_mse_l1.argtypes = [fp, fp, ci, ci, ci, ci, ci, ci, ci, fp, fp, fp, vp]
    cf, cll = ctypes.c_float, ctypes.c_longlong
    L.nint_fuse_inputs.argtypes = [fp, fp, fp, fp, fp, ci, cll, ci, ci, ci, ci, ci, ci, fp, vp]
    L.nint_adam_step.argtypes = [fp, fp, fp, fp, cll, cf, cf, cf, cf, ci, cf, vp]
    L.nint_adam_step_dev.argtypes = [fp, fp, fp, fp, cll, fp, cf, cf, cf, cf, vp]
    L.nint_dp_allreduce_adam.argtypes = [ctypes.POINTER(vp), cll, cll, ci, ci, ctypes.c_uint, fp, fp, fp, cll, fp, cf, cf, cf, cf, vp]
    L.nint_fuse_inputs_bank.argtypes = [fp, fp, fp, fp, fp, ci, cll, ci, ci, ci, ci, ci, ci, ci, ci, ci, fp, vp]
    L.nint_fuse_inputs_adjoint.argtypes = [fp, fp, cll, ci, ci, ci, ci, ci, ci, ci, fp, fp, fp, vp]
    L.nint_loss_mse_l1_bank.argtypes = [fp, fp, cll, fp, ci, ci, ci, ci, ci, ci, ci, ci, fp, fp, fp, vp]
    L.nint_pick_tile.argtypes = [ci, ci, ctypes.POINTER(ci), ctypes.POINTER(ci)]
    for name in EXPORTS:
        getattr(L, name)  # raises AttributeError if the library does not export what nint.h declares
    _lib = L
    return L


def check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what}: {load().nint_last_error().decode()}")


def ptr(t):
    """device pointer of a tensor (or None) as a ctypes void pointer"""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    """torch's current stream ON `device` (not on the current device) as a ctypes pointer"""
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def on_device(device):
    """Context manager: libnint calls launch on the CUDA runtime's current device, so every call that touches
    `device`'s memory runs inside this guard (a model on cuda:1 with current device 0 would otherwise launch on GPU 0
    against GPU 1 pointers)."""
    import torch
    return torch.cuda.device(device)


def pick_tile(height, width):
    tw, th = ctypes.c_int(), ctypes.c_int()
    check(load().nint_pick_tile(height, width, ctypes.byref(tw), ctypes.byref(th)), "nint_pick_tile")
    return tw.value, th.value
