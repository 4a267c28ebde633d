"""ctypes binding of liblbbnn.so (include/lbbnn.h).  No torch types cross this boundary: tensors are
passed as raw device pointers + sizes, the stream as the raw cudaStream_t handle.

There is NO CPU fallback: if the library is missing this module raises at import, and every wrapper
rejects non-CUDA tensors.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblbbnn.so")

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: the CUDA extension has not been built "
        "(run `python bayesian-neural-nets_b200/build.py` or __graft_entry__.build()). "
        "lbbnn has no CPU or eager-PyTorch fallback.")

lib = C.CDLL(LIB_PATH)

VAR_REFERENCE, VAR_EXACT = 0, 1
FLAG_SAMPLE, FLAG_RELU, FLAG_KL, FLAG_ACCUMULATE, FLAG_MASK_DX, FLAG_MOMENTS = 1, 2, 4, 8, 16, 32
PACK_PAIR, PACK_SQUARE, PACK_SCALE = 0, 1, 2
MF_SAMPLE, MF_MEDIMEAN, MF_JOINTMEAN = 0, 1, 2
MF_FLAG_LOGPROBS, MF_FLAG_LP_ON_WS, MF_FLAG_EXACT_GAMMA, MF_FLAG_EXACT_WPRIOR, MF_FLAG_EXACT_GPRIOR = 1, 2, 4, 8, 16


class Priors(C.Structure):
    _fields_ = [("mu", C.c_float), ("sigma", C.c_float), ("alpha", C.c_float),
                ("bias_mu", C.c_float), ("bias_sigma", C.c_float)]


class Layer(C.Structure):
    _fields_ = [("weight_mu", C.c_void_p), ("weight_rho", C.c_void_p), ("lambdal", C.c_void_p),
                ("bias_mu", C.c_void_p), ("bias_rho", C.c_void_p), ("z", C.c_void_p),
                ("in_features", C.c_int64), ("out_features", C.c_int64), ("z_kl", C.c_void_p)]


class LayerGrads(C.Structure):
    _fields_ = [("weight_mu", C.c_void_p), ("weight_rho", C.c_void_p), ("lambdal", C.c_void_p),
                ("bias_mu", C.c_void_p), ("bias_rho", C.c_void_p), ("z", C.c_void_p), ("z_kl", C.c_void_p)]


class Noise(C.Structure):
    _fields_ = [("eps", C.c_void_p), ("seed", C.c_uint64), ("stream_id", C.c_uint64),
                ("step_dev", C.c_void_p), ("step_stride", C.c_uint64)]


FLOW_MAX_T, FLOW_MAX_HIDDEN = 8, 6
FLOW_RNVP, FLOW_IAF = 0, 1


class FlowLinear(C.Structure):
    _fields_ = [("W", C.c_void_p), ("b", C.c_void_p), ("in_", C.c_int), ("out", C.c_int)]


class FlowTransform(C.Structure):
    _fields_ = [("hidden", FlowLinear * FLOW_MAX_HIDDEN), ("shift", FlowLinear), ("scale", FlowLinear)]


class Flow(C.Structure):
    _fields_ = [("kind", C.c_int), ("dim", C.c_int), ("n_transforms", C.c_int), ("n_hidden", C.c_int),
                ("t", FlowTransform * FLOW_MAX_T)]


class FlowLinearGrad(C.Structure):
    _fields_ = [("dW", C.c_void_p), ("db", C.c_void_p)]


class FlowTransformGrads(C.Structure):
    _fields_ = [("hidden", FlowLinearGrad * FLOW_MAX_HIDDEN), ("shift", FlowLinearGrad), ("scale", FlowLinearGrad)]


class FlowGrads(C.Structure):
    _fields_ = [("row_stride", C.c_int64), ("t", FlowTransformGrads * FLOW_MAX_T)]


class AdamLayerState(C.Structure):
    _fields_ = [("exp_avg", C.c_void_p * 5), ("exp_avg_sq", C.c_void_p * 5), ("coef", C.c_void_p),
                ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float)]


class DpLayer(C.Structure):
    _fields_ = [("world", C.c_int), ("rank", C.c_int), ("raw_mc", C.c_void_p), ("weight_mu_mc", C.c_void_p),
                ("weight_rho_mc", C.c_void_p), ("lambdal_mc", C.c_void_p), ("bias_mu_mc", C.c_void_p), ("bias_rho_mc", C.c_void_p)]


class MnfAux(C.Structure):
    _fields_ = [("in_features", C.c_int64), ("out_features", C.c_int64)] + [
        (n, C.c_void_p) for n in ("q0_mean", "q0_log_var", "z0", "r0_c", "r0_b1", "r0_b2", "z2", "M0", "V", "eps_r", "z_b")]


class MnfAuxGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("d_q0_mean", "d_q0_log_var", "d_z0", "d_r0_c", "d_r0_b1", "d_r0_b2", "d_z2",
                                          "d_z_b", "dM0", "dV")]


STEP_MAX_LAYERS = 8


class StepLayer(C.Structure):
    _fields_ = [("in_features", C.c_int64), ("out_features", C.c_int64), ("off_weight_mu", C.c_int64),
                ("off_weight_rho", C.c_int64), ("off_lambdal", C.c_int64), ("off_bias_mu", C.c_int64),
                ("off_bias_rho", C.c_int64), ("eps", C.c_void_p), ("priors", Priors), ("var_mode", C.c_int)]


class StepDp(C.Structure):
    _fields_ = [("world", C.c_int), ("rank", C.c_int), ("flat_mc", C.c_void_p), ("ws_mc", C.c_void_p),
                ("signal", C.c_void_p * 8), ("klx", C.c_void_p * 8), ("epoch", C.c_void_p), ("use_p2p", C.c_int),
                ("flat_peer", C.c_void_p * 8), ("ws_peer", C.c_void_p * 8)]


class Step(C.Structure):
    _fields_ = [("n_layers", C.c_int), ("batch", C.c_int64), ("layer", StepLayer * STEP_MAX_LAYERS),
                ("flat", C.c_void_p), ("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p), ("grad", C.c_void_p),
                ("x", C.c_void_p), ("y", C.c_void_p), ("step_dev", C.c_void_p), ("seed", C.c_uint64),
                ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("kl_scale", C.c_float), ("stats", C.c_void_p), ("dp", C.POINTER(StepDp))]


_P, _I64, _U64, _INT, _F, _SZ = C.c_void_p, C.c_int64, C.c_uint64, C.c_int, C.c_float, C.c_size_t

# name -> (restype, argtypes); kept in one table so tests can check every header symbol is bound
SIGNATURES = {
    "lbbnn_last_error": (C.c_char_p, []),
    "lbbnn_abi_version": (_INT, []),
    "lbbnn_device_ok": (_INT, []),
    "lbbnn_philox_normal": (_INT, [_P, _I64, _U64, _U64, _P]),
    "lbbnn_philox_uniform": (_INT, [_P, _I64, _U64, _U64, _P]),
    "lbbnn_philox_normal_ex": (_INT, [_P, _I64, C.POINTER(Noise), _P]),
    "lbbnn_lrt_f32_workspace_bytes": (_SZ, [_I64, _I64, _I64]),
    "lbbnn_lrt_f32_mv_bytes": (_SZ, [_I64, _I64]),
    "lbbnn_lrt_f32_fwd": (_INT, [C.POINTER(Layer), _P, _I64, C.POINTER(Noise), C.POINTER(Priors), _INT, _INT,
                                 _P, _P, _P, _P, _P, _SZ, _P]),
    "lbbnn_lrt_f32_fwd_ex": (_INT, [C.POINTER(Layer), _P, _I64, C.POINTER(Noise), C.POINTER(Priors), _INT, _INT,
                                    _P, _P, _P, _P, _P, _I64, _U64, _P, _SZ, _P]),
    "lbbnn_lrt_sample_expand": (_INT, [_P, _P, _I64, _I64, _INT, C.POINTER(Noise), _U64, _INT, _P, _P]),
    "lbbnn_lrt_f32_bwd_params": (_INT, [C.POINTER(Layer), _P, _I64, _P, _P, C.POINTER(Priors), _INT, _INT, _P, _F,
                                        C.POINTER(LayerGrads), _P, _SZ, _P]),
    "lbbnn_lrt_f32_bwd_input": (_INT, [C.POINTER(Layer), _P, _I64, _P, _P, C.POINTER(Priors), _INT, _INT, _P, _P,
                                       _P, _SZ, _P]),
    "lbbnn_lrt_f32_prologue": (_INT, [C.POINTER(Layer), C.POINTER(Priors), _INT, _INT, _P, _P, _P, _P, _SZ, _P]),
    "lbbnn_lrt_f32_finalize": (_INT, [C.POINTER(Layer), _P, _P, _P, C.POINTER(Priors), _INT, _INT, _P, _F,
                                      C.POINTER(LayerGrads), _P]),
    "lbbnn_lrt_f32_finalize_adam": (_INT, [C.POINTER(Layer), _P, _P, _P, C.POINTER(Priors), _INT, _INT, _P, _F,
                                           C.POINTER(AdamLayerState), _P]),
    "lbbnn_adam_prepare": (_INT, [_P, _F, _F, _F, _P, _P]),
    "lbbnn_tc_dual_gemm_raw": (_INT, [_P, _P, _P, _P, _I64, _I64, _I64, _P, _P, _P]),
    "lbbnn_tc_lrt_fwd": (_INT, [_P, _P, _P, _P, _I64, _I64, _I64, _P, _P, C.POINTER(Noise), _INT,
                                _P, _P, _P, _P, _P, _P, _P]),
    "lbbnn_tc_lrt_bwd_input": (_INT, [_P, _P, _P, _P, _I64, _I64, _I64, _P, _P, _INT, _P, _P, _P, _P, _P]),
    "lbbnn_bf16_pack": (_INT, [_P, _P, _INT, _I64, _I64, _P, _P, _P, _P, _P]),
    "lbbnn_lrt_bf16_prologue_workspace_bytes": (_SZ, [_I64, _I64]),
    "lbbnn_lrt_bf16_prologue": (_INT, [C.POINTER(Layer), C.POINTER(Priors), _INT, _P, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "lbbnn_lrt_bf16_prologue_kl_parts": (_SZ, [_I64, _I64]),
    "lbbnn_lrt_bf16_prologue_parts": (_INT, [C.POINTER(Layer), C.POINTER(Priors), _INT, _P, _P, _P, _P, _P, _SZ, _P]),
    "lbbnn_tc_lrt_bwd_input_small_workspace_bytes": (_SZ, [_I64, _I64]),
    "lbbnn_tc_lrt_bwd_input_small": (_INT, [_P, _P, _P, _P, _I64, _I64, _I64, _P, _P, _INT, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "lbbnn_tc_lrt_fwd_small": (_INT, [_P, _P, _P, _P, _I64, _I64, _I64, _P, _P, C.POINTER(Noise), _INT, _P, _P, _P]),
    "lbbnn_tc_dual_gemm_raw_small": (_INT, [_P, _P, _P, _P, _I64, _I64, _I64, _P, _P, _P]),
    "lbbnn_tc_dual_gemm_raw_ex": (_INT, [_P, _P, _P, _P, _I64, _I64, _I64, _INT, _INT, _P, _P, _P]),
    "lbbnn_tc_colsum_part_floats": (_SZ, [_I64, _I64]),
    "lbbnn_tc_colsum_reduce": (_INT, [_P, _I64, _I64, _P, _P]),
    "lbbnn_tc_lrt_bwd_input_mn": (_INT, [_P, _P, _P, _P, _I64, _I64, _I64, _P, _P, _INT, _P, _P, _P, _P]),
    "lbbnn_tc_lrt_dw_adam": (_INT, [_P, _P, _P, _P, C.POINTER(Layer), _I64, C.POINTER(Priors), _INT, _F,
                                    C.POINTER(AdamLayerState), _P]),
    "lbbnn_tc_lrt_dw_adam_kl_parts": (_SZ, []),
    "lbbnn_tc_lrt_dw_adam_next": (_INT, [_P, _P, _P, _P, C.POINTER(Layer), _I64, C.POINTER(Priors), _INT, _F,
                                         C.POINTER(AdamLayerState), _P, _P, _P, _P]),
    "lbbnn_lrt_kl_finalize": (_INT, [_P, _I64, C.POINTER(Layer), C.POINTER(Priors), _P, _P]),
    "lbbnn_lrt_f32_finalize_adam_bias": (_INT, [C.POINTER(Layer), _P, C.POINTER(Priors), _INT, _F, C.POINTER(AdamLayerState), _P]),
    "lbbnn_lrt_f32_finalize_adam_dp": (_INT, [C.POINTER(Layer), C.POINTER(DpLayer), C.POINTER(Priors), _INT, _INT, _F,
                                              C.POINTER(AdamLayerState), _P]),
    "lbbnn_colsum2_workspace_bytes": (_SZ, [_I64, _I64]),
    "lbbnn_colsum2": (_INT, [_P, _P, _INT, _I64, _I64, _P, _P, _SZ, _P]),
    "lbbnn_linear_f32_fwd": (_INT, [_P, _P, _P, _I64, _I64, _I64, _INT, _P, _P, _SZ, _P]),
    "lbbnn_linear_f32_bwd_params": (_INT, [_P, _P, _I64, _I64, _I64, _P, _P, _P, _SZ, _P]),
    "lbbnn_linear_f32_bwd_input": (_INT, [_P, _P, _P, _I64, _I64, _I64, _INT, _P, _P, _SZ, _P]),
    "lbbnn_mf_workspace_bytes": (_SZ, [_I64]),
    "lbbnn_mf_gamma_sample": (_INT, [_P, _P, _I64, C.POINTER(Noise), _INT, _F, _P, _P]),
    "lbbnn_mf_gamma_sample_bwd": (_INT, [_P, _P, _P, _P, _I64, _F, _P, _P]),
    "lbbnn_mf_sample_fwd": (_INT, [_P, _P, _P, _P, _P, _P, _I64, C.POINTER(Noise), _INT, _INT, _P, _P, _P, _SZ, _P]),
    "lbbnn_mf_sample_fwd_ticket": (_INT, [_P, _P, _P, _P, _P, _P, _I64, C.POINTER(Noise), _INT, _INT, _P, _P, _P, _SZ, _P, _P]),
    "lbbnn_mf_sample_bwd_ticket": (_INT, [_P, _P, _P, _P, _P, _I64, C.POINTER(Noise), _INT, _P, _P, _P, _P, _P, _P, _P, _P, _SZ,
                                          _P, _P]),
    "lbbnn_mf_sample_predict": (_INT, [C.POINTER(Layer), C.POINTER(Noise), C.POINTER(Noise), C.POINTER(Noise), _P, _P, _P]),
    "lbbnn_mc_accumulate": (_INT, [_P, _I64, _I64, _P, _P, _P, _P]),
    "lbbnn_mc_sample": (_INT, [C.POINTER(Layer), _INT, _P, _U64, _U64, _U64, _P, _P, _P]),
    "lbbnn_linear_f32_batched": (_INT, [_P, _I64, _P, _P, _INT, _I64, _I64, _I64, _INT, _P, _P]),
    "lbbnn_mc_accumulate_batched": (_INT, [_P, _INT, _I64, _I64, _P, _P, _P, _P]),
    "lbbnn_tf32_split": (_INT, [_P, _I64, _P, _P, _P]),
    "lbbnn_lrt_mc_epilogue": (_INT, [_P, _I64, _P, _I64, _P, _P, _I64, _I64, _INT, C.POINTER(Noise), _U64, _INT, _P, _P,
                                     _P, _P, _P, _P, _P]),
    "lbbnn_tf32_split_rows": (_INT, [_P, _I64, _I64, _I64, _INT, _P, _P, _P, _P, _P, _P]),
    "lbbnn_mc_head_accumulate": (_INT, [_P, _I64, _P, _P, _INT, _I64, _I64, _I64, _P, _P, _P, _P]),
    "lbbnn_mc_prepare": (_INT, [C.POINTER(Layer), _P, _P, _P, _P]),
    "lbbnn_mc_sample_split": (_INT, [C.POINTER(Layer), _INT, _P, _U64, _U64, _U64, _INT, _P, _P, _P, _P]),
    "lbbnn_tc_linear_tf32x3": (_INT, [_P, _P, _I64, _I64, _P, _P, _P, _I64, _I64, _I64, _I64, _INT, _P, _P, _P,
                                      _I64, _I64, _P]),
    "lbbnn_mf_sample_bwd": (_INT, [_P, _P, _P, _P, _P, _I64, C.POINTER(Noise), _INT, _P, _P, _P, _P, _P, _P, _P,
                                   _P, _SZ, _P]),
    "lbbnn_mf_prior_fwd": (_INT, [_P] * 11 + [C.POINTER(Noise), _INT, _I64, C.c_double, _P, _P, _P, _P]),
    "lbbnn_mf_prior_bwd": (_INT, [_P] * 13 + [_INT, _I64, C.c_double] + [_P] * 9 + [_P]),
    "lbbnn_mf_prior_bwd_tau": (_INT, [_P] * 13 + [_INT, _I64, C.c_double] + [_P] * 13 + [_P]),
    "lbbnn_flow_save_floats": (_SZ, [C.POINTER(Flow), _I64]),
    "lbbnn_flow_fwd": (_INT, [C.POINTER(Flow), _P, _I64, _P, C.POINTER(Noise), _P, _P, _P, _P]),
    "lbbnn_flow_bwd": (_INT, [C.POINTER(Flow), C.POINTER(FlowGrads), _I64, _P, C.POINTER(Noise), _P, _P, _P, _P, _P]),
    "lbbnn_mnf_aux_save_floats": (_SZ, [_I64]),
    "lbbnn_mnf_aux_kl_fwd": (_INT, [C.POINTER(MnfAux), _P, _P, _P, _P]),
    "lbbnn_mnf_aux_kl_bwd": (_INT, [C.POINTER(MnfAux), _P, _P, C.POINTER(MnfAuxGrads), _P]),
    "lbbnn_mnf_draw": (_INT, [_P, _P, C.POINTER(Noise), _I64, _I64, _P, _P, C.POINTER(Noise), _I64, _P, _P]),
    "lbbnn_mnf_draw_bwd": (_INT, [_P, _P, _P, _I64, _I64, _INT, _P, _P, _P, _P, _P, _P]),
    "lbbnn_mnf_kl_combine": (_INT, [_P, _P, _P, _P, _P, _P]),
    "lbbnn_mnf_bwd_rows": (_INT, [_P, _F, _P, _P, _P, _P, _I64, _P, _P]),
    "lbbnn_lrt_step_workspace_bytes": (_SZ, [C.POINTER(Step)]),
    "lbbnn_lrt_step_raw_floats": (_SZ, [C.POINTER(Step)]),
    "lbbnn_lrt_step_f32": (_INT, [C.POINTER(Step), _INT, _P, _SZ, _P]),
    "lbbnn_lrt_step_profile": (_INT, [_P]),
    "lbbnn_lrt_step_describe": (_INT, [C.POINTER(Step), C.c_char_p, _SZ]),
    "lbbnn_logsoftmax_nll_f32": (_INT, [_P, _P, _I64, _I64, _P, _P, _P, _F, _P, _P, _SZ, _P]),
    "lbbnn_adam_f32": (_INT, [_P, _P, _P, _P, _I64, _F, _F, _F, _F, _P, _P, _P]),
    "lbbnn_adam_multi_f32": (_INT, [_P, _INT, _I64, _F, _F, _F, _F, _P, _P, _P]),
    "lbbnn_adam_multi_step_f32": (_INT, [_P, _INT, _I64, _F, _F, _F, _F, _P, _P, _P]),
    "lbbnn_nll_kl_objective_f32": (_INT, [_P, _P, _I64, _I64, _P, _P, _INT, _F, _P, _P, _P]),
    "lbbnn_adam_pack_f32": (_INT, [_P, _INT, _I64, _I64, _P]),
    "lbbnn_adam_multi_dp_f32": (_INT, [_P, _INT, _I64, _I64, _P, _P, _I64, _F, _F, _F, _F, _P, _P, _INT, _P]),
    "lbbnn_counter_inc": (_INT, [_P, _P]),
    "lbbnn_adamw_f32": (_INT, [_P, _P, _P, _P, _I64, _F, _F, _F, _F, _F, _P, _P, _P]),
    "lbbnn_vd_workspace_bytes": (_SZ, [_I64, _I64, _I64]),
    "lbbnn_vd_gemm_launches": (_INT, [_I64, _I64, _I64]),
    "lbbnn_vd_fwd": (_INT, [_P, _P, _P, _I64, _I64, _I64, C.POINTER(Noise), _INT, _P, _P, _P, _P, _SZ, _P]),
    "lbbnn_vd_bwd": (_INT, [_P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _INT, _P, _P, _P, _P, _SZ, _P]),
    "lbbnn_vd_kl": (_INT, [_P, _I64, _P, _INT, _P, _F, _P]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)   # AttributeError here = header/library mismatch: fail loudly
    _fn.restype = _res
    _fn.argtypes = _args


class LbbnnError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        raise LbbnnError(f"liblbbnn error {rc}: {lib.lbbnn_last_error().decode()}")


def ptr(t, dtype=torch.float32, allow_none=False):
    """Raw device pointer of a contiguous CUDA tensor on the CURRENT device (the only kind the library accepts: every
    wrapper launches on the current device's current stream, so a tensor living elsewhere would be dereferenced by the
    wrong GPU).  ptr(t, True) is shorthand for fp32 with None allowed."""
    if isinstance(dtype, bool):
        dtype, allow_none = torch.float32, dtype
    if t is None:
        if allow_none:
            return None
        raise LbbnnError("required tensor is None")
    if not t.is_cuda:
        raise LbbnnError("lbbnn kernels take CUDA tensors only (no CPU fallback); got a CPU tensor")
    if t.device.index != torch.cuda.current_device():
        raise LbbnnError(f"tensor lives on cuda:{t.device.index} but the current device is cuda:{torch.cuda.current_device()}; "
                         "wrap the call in torch.cuda.device(tensor.device) (kernels launch on the current device's stream)")
    if t.dtype != dtype:
        raise LbbnnError(f"expected {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise LbbnnError("tensor must be contiguous")
    return t.data_ptr()


def current_stream():
    return torch.cuda.current_stream().cuda_stream


_device_checked = set()


def require_device():
    """Raises unless the current CUDA device is a compute-capability-10.x GPU (checked once per device)."""
    if not torch.cuda.is_available():
        raise LbbnnError("no CUDA device: lbbnn runs on B200 (sm_100a) only and has no CPU fallback")
    dev = torch.cuda.current_device()
    if dev in _device_checked:
        return
    if not lib.lbbnn_device_ok():
        raise LbbnnError("the current CUDA device is not compute capability 10.x; liblbbnn is sm_100a-only")
    _device_checked.add(dev)


# ---- workspace: one growable buffer per (device, stream) -------------------------------------------
_workspaces = {}


def workspace(nbytes, device):
    key = (device.index if device.index is not None else torch.cuda.current_device(), current_stream())
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        if torch.cuda.is_current_stream_capturing():
            raise LbbnnError("workspace would have to grow during CUDA-graph capture; run one eager step first")
        ws = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def lrt_workspace_bytes(batch, in_features, out_features):
    return int(lib.lbbnn_lrt_f32_workspace_bytes(batch, in_features, out_features))


def lrt_mv_bytes(in_features, out_features):
    return int(lib.lbbnn_lrt_f32_mv_bytes(in_features, out_features))


def make_layer(weight_mu, weight_rho, lambdal, bias_mu, bias_rho, z=None, z_kl=None):
    out_f, in_f = weight_mu.shape
    return Layer(ptr(weight_mu), ptr(weight_rho), ptr(lambdal), ptr(bias_mu), ptr(bias_rho),
                 ptr(z, allow_none=True), in_f, out_f, ptr(z_kl, allow_none=True))


# While a whole-step CUDA graph is being warmed up / captured (engine.GraphedTrainer), every native-noise call of the
# drop-in modules adds  *step * GRAPH_NOISE_STRIDE  to its Philox stream: the stream ids are Python integers baked into
# the captured launches, the device step counter is what makes each replay draw fresh noise.
GRAPH_NOISE_STRIDE = 0x9E3779B1
_graph_noise_step = None


class graph_noise:
    def __init__(self, step_tensor):
        self.step = step_tensor

    def __enter__(self):
        global _graph_noise_step
        self.prev, _graph_noise_step = _graph_noise_step, self.step
        return self

    def __exit__(self, *exc):
        global _graph_noise_step
        _graph_noise_step = self.prev


# Data-parallel training (engine.GraphedTrainer with a process group): the noise that belongs to the minibatch ROWS -- the
# activation eps of the LRT / MNF layers -- must differ between ranks, while the draws that depend on the parameters only are
# shared.  While a trainer holds row_noise_rank(rank), lrt.py adds 0x9E3779B97F4A7C15 * rank to the seed of the activation
# noise (the convention of the LRT trainers) and nothing else.
_row_seed_offset = 0


class row_noise_rank:
    def __init__(self, rank):
        self.offset = (0x9E3779B97F4A7C15 * int(rank)) & (2 ** 64 - 1)

    def __enter__(self):
        global _row_seed_offset
        self.prev, _row_seed_offset = _row_seed_offset, self.offset
        return self

    def __exit__(self, *exc):
        global _row_seed_offset
        _row_seed_offset = self.prev


def row_noise_seed(seed):
    return (seed + _row_seed_offset) & (2 ** 64 - 1)


def make_noise(eps=None, seed=0, stream_id=0, step_dev=None, step_stride=0):
    if eps is None and step_dev is None and _graph_noise_step is not None:
        step_dev, step_stride = _graph_noise_step, GRAPH_NOISE_STRIDE
    return Noise(ptr(eps, allow_none=True), seed & (2 ** 64 - 1), stream_id & (2 ** 64 - 1),
                 ptr(step_dev, torch.int64, allow_none=True), step_stride)


def philox_normal(shape, seed, stream_id, device="cuda"):
    """Materialise the native N(0,1) noise of stream (seed, stream_id) -- what a fused kernel draws."""
    require_device()
    out = torch.empty(shape, dtype=torch.float32, device=device)
    check(lib.lbbnn_philox_normal(ptr(out), out.numel(), seed, stream_id, current_stream()))
    return out


def philox_uniform(shape, seed, stream_id, device="cuda"):
    require_device()
    out = torch.empty(shape, dtype=torch.float32, device=device)
    check(lib.lbbnn_philox_uniform(ptr(out), out.numel(), seed, stream_id, current_stream()))
    return out


# ---- bf16 tensor-core path ----------------------------------------------------------------------------
BF16 = torch.bfloat16


def bf16_pack(a, b, op, transposed=True):
    """fp32 (rows, cols) -> (bf16 a, bf16 f(a,b)) and, if asked, their (cols, rows) transposes."""
    require_device()
    rows, cols = a.shape
    o1 = torch.empty(rows, cols, dtype=BF16, device=a.device)
    o2 = torch.empty(rows, cols, dtype=BF16, device=a.device)
    o1t = torch.empty(cols, rows, dtype=BF16, device=a.device) if transposed else None
    o2t = torch.empty(cols, rows, dtype=BF16, device=a.device) if transposed else None
    check(lib.lbbnn_bf16_pack(ptr(a), ptr(b, allow_none=True), op, rows, cols, ptr(o1, BF16), ptr(o2, BF16),
                              ptr(o1t, BF16, allow_none=True), ptr(o2t, BF16, allow_none=True), current_stream()))
    return o1, o2, o1t, o2t


def tc_dual_gemm_raw(a1, a2, b1, b2, a_mn=False, b_mn=False):
    """D1 = A1 @ B1.T, D2 = A2 @ B2.T (bf16 in, fp32 out) on tcgen05.  K-major operands are (rows, K) tensors; with
    a_mn / b_mn the operand is passed as the (K, rows) tensor it is the transpose of (read in place, "MN-major")."""
    require_device()
    k, m = a1.shape if a_mn else a1.shape[::-1]
    n = b1.shape[1] if b_mn else b1.shape[0]
    d1 = torch.empty(m, n, dtype=torch.float32, device=a1.device)
    d2 = torch.empty(m, n, dtype=torch.float32, device=a1.device)
    check(lib.lbbnn_tc_dual_gemm_raw_ex(ptr(a1, BF16), ptr(a2, BF16), ptr(b1, BF16), ptr(b2, BF16), m, n, k,
                                        int(bool(a_mn)), int(bool(b_mn)), ptr(d1), ptr(d2), current_stream()))
    return d1, d2
