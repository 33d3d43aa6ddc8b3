"""ctypes binding of libmobody_b200.so (include/mobody_b200.h).

The product has no CPU or eager-PyTorch fallback: if the shared library is missing or a CUDA
device is not available, calls raise immediately.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# MOBODY_B200_LIB selects another build of the same library (kernel A/B experiments, scripts/build_variant.py)
LIB_PATH = os.environ.get("MOBODY_B200_LIB") or os.path.join(_HERE, "libmobody_b200.so")

N_DYN_LAYERS = 13
DYN_LAYER_NAMES = ("zs1", "zs2", "zs3", "za_src1", "za_src2", "za_trg1", "za_trg2",
                   "transition1", "transition2", "transition3",
                   "reward_model1", "reward_model2", "reward_model3")
# fp32: CUDA-core kernel; bf16x2: tcgen05 hi+lo split, inside the 1e-4 bound (default); fp16: tcgen05 single pass, inside the
# stated looser bound 5e-3; bf16x2_wide: bf16x2's arithmetic on 64-row tiles for 65 <= S <= 128; bf16x2_t64: the same 64-row
# kernel for the S <= 64 shapes bf16x2 refuses (A > 16 or 2S+A > 96: Adroit).  Both are opt-in: "auto" keeps fp32 for the
# shapes bf16x2 refuses.  The library's single-pass bf16 mode (code 2, measured 1.6e-2) is outside every stated bound: it is a
# kernel-development diagnostic and is not offered here.
PREC = {"fp32": 0, "bf16x2": 1, "fp16": 3, "bf16x2_wide": 4, "bf16x2_t64": 5}
# the general modes, which take the small shapes every test and the benchmark sweep; bf16x2_wide and bf16x2_t64 do not
ENABLED_PRECISIONS = ("fp32", "bf16x2", "fp16")
# shapes the tensor-core modes take (MOBODY_TC_* in include/mobody_b200.h): S <= 64, A <= 16, 2S+A <= the mode's limit
TC_MAX_S, TC_MAX_A, TC_MAX_SAS = 64, 16, {"bf16x2": 96, "fp16": 112}
# shapes of bf16x2_wide (MOBODY_TC_WIDE_*): TC_WIDE_MIN_S <= S <= TC_WIDE_MAX_S, A <= TC_WIDE_MAX_A
TC_WIDE_MIN_S, TC_WIDE_MAX_S, TC_WIDE_MAX_A = 65, 128, 32
# shapes of bf16x2_t64 (MOBODY_TC_T64_*): 2 <= S <= TC_T64_MAX_S, A <= TC_T64_MAX_A, and a shape bf16x2 refuses
TC_T64_MAX_S, TC_T64_MAX_A = 64, 32
ABI_VERSION = 2
TC_TRAIN_MIN_ROWS = 1280   # MOBODY_TC_TRAIN_MIN_ROWS: mobody_train_step runs on tcgen05 GEMM tiles from this many batch rows
KEEP_U8_ZERO, KEEP_F32_LE, KEEP_F32_LT, KEEP_U8_VALID = 0, 1, 2, 3


class DynParams(C.Structure):
    _fields_ = [("w", C.c_void_p * N_DYN_LAYERS), ("b", C.c_void_p * N_DYN_LAYERS)]


class MlpParams(C.Structure):
    _fields_ = [("w", C.c_void_p * 3), ("b", C.c_void_p * 3)]


class StepDesc(C.Structure):
    _fields_ = [
        ("precision", C.c_int), ("B", C.c_int), ("S", C.c_int), ("A", C.c_int), ("obs_ld", C.c_int), ("act_ld", C.c_int),
        ("n_rows_dev", C.c_void_p), ("row_ids", C.c_void_p),
        ("obs", C.c_void_p), ("act", C.c_void_p),
        ("policy", C.POINTER(MlpParams)), ("max_action", C.c_float),
        ("dyn", C.POINTER(DynParams)), ("dyn_pack", C.c_void_p), ("policy_pack", C.c_void_p),
        ("use_trg", C.c_int), ("use_penalty", C.c_int), ("penalty_coef", C.c_float), ("term_kind", C.c_int),
        ("eps", C.c_void_p), ("idx", C.c_void_p), ("elites", C.c_void_p), ("n_elites", C.c_int),
        ("seed", C.c_ulonglong), ("step", C.c_uint), ("row0", C.c_ulonglong),
        ("act_out", C.c_void_p), ("next_obs", C.c_void_p), ("reward", C.c_void_p), ("raw_reward", C.c_void_p),
        ("penalty", C.c_void_p), ("terminal", C.c_void_p), ("mean", C.c_void_p),
    ]


class RolloutDesc(C.Structure):
    _fields_ = [
        ("step", StepDesc), ("T", C.c_int), ("filter_bad_rollout", C.c_int), ("env_filter", C.c_float),
        ("eps_all", C.c_void_p), ("idx_all", C.c_void_p),
        ("obss", C.c_void_p), ("acts", C.c_void_p), ("nexts", C.c_void_p), ("rews", C.c_void_p), ("pens", C.c_void_p),
        ("terms", C.c_void_p), ("row_ids", C.c_void_p), ("counts", C.c_void_p), ("pos", C.c_void_p), ("scratch", C.c_void_p),
        ("stats", C.c_void_p), ("ticket", C.c_void_p), ("packed", C.c_void_p),
    ]


class ModelEvalDesc(C.Structure):
    _fields_ = [
        ("step", StepDesc), ("H", C.c_int), ("gamma", C.c_double), ("workspace", C.c_void_p), ("workspace_bytes", C.c_longlong),
        ("ret", C.c_void_p), ("ret_disc", C.c_void_p), ("length", C.c_void_p), ("counts", C.c_void_p),
    ]


class PeerDesc(C.Structure):
    _fields_ = [("world", C.c_int), ("rank", C.c_int), ("base", C.c_void_p * 8), ("multicast", C.c_void_p), ("cap_rows", C.c_longlong), ("W", C.c_int),
                ("epoch", C.c_uint), ("ctas", C.c_int)]


class SampleJob(C.Structure):
    _fields_ = [("rows", C.c_void_p), ("n", C.c_longlong), ("size", C.c_uint), ("draw", C.c_uint), ("seed", C.c_ulonglong),
                ("out", C.c_void_p)]


class MlpState(C.Structure):
    _fields_ = [("w", C.c_void_p * 3), ("b", C.c_void_p * 3)]


class TrainDesc(C.Structure):
    _fields_ = [
        ("rows", C.c_void_p), ("N", C.c_int), ("n_true", C.c_int), ("S", C.c_int), ("A", C.c_int), ("row_width", C.c_int),
        ("policy", MlpState), ("q1", MlpState), ("q2", MlpState), ("q1_target", MlpState), ("q2_target", MlpState),
        ("policy_m", MlpState), ("policy_v", MlpState), ("q1_m", MlpState), ("q1_v", MlpState), ("q2_m", MlpState), ("q2_v", MlpState),
        ("t_q", C.c_int), ("t_pi", C.c_int),
        ("gamma", C.c_float), ("tau", C.c_float), ("critic_lr", C.c_float), ("actor_lr", C.c_float), ("weight", C.c_float),
        ("bc_coef", C.c_float), ("max_action", C.c_float),
        ("nsplit", C.c_int), ("workspace", C.c_void_p), ("workspace_bytes", C.c_longlong), ("scalars_out", C.c_void_p),
    ]


class TrainExDesc(C.Structure):
    _fields_ = [
        ("base", TrainDesc), ("advantage", C.c_int), ("scale_q", C.c_int), ("q_weighted", C.c_int),
        ("value", MlpState), ("value_m", MlpState), ("value_v", MlpState), ("t_v", C.c_int),
    ]


class ClassifierDesc(C.Structure):
    _fields_ = [
        ("rows", C.c_void_p), ("N", C.c_int), ("S", C.c_int), ("A", C.c_int), ("row_width", C.c_int),
        ("label", C.c_void_p), ("noise_sas", C.c_void_p), ("noise_sa", C.c_void_p),
        ("noise_std", C.c_float), ("seed", C.c_ulonglong), ("draw", C.c_uint),
        ("sas", MlpState), ("sa", MlpState), ("sas_m", MlpState), ("sas_v", MlpState), ("sa_m", MlpState), ("sa_v", MlpState),
        ("t", C.c_int), ("lr", C.c_float), ("nsplit", C.c_int),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_longlong), ("scalars_out", C.c_void_p),
    ]


class DynState(C.Structure):
    _fields_ = [("w", C.c_void_p * N_DYN_LAYERS), ("b", C.c_void_p * N_DYN_LAYERS)]


class DynFitDesc(C.Structure):
    _fields_ = [
        ("S", C.c_int), ("A", C.c_int), ("B", C.c_int), ("use_trg", C.c_int),
        ("obs", C.c_void_p), ("act", C.c_void_p), ("next_obs", C.c_void_p), ("reward", C.c_void_p), ("member_stride", C.c_longlong),
        ("eps_latent", C.c_void_p), ("eps_next", C.c_void_p), ("seed", C.c_ulonglong), ("draw", C.c_uint),
        ("encoder_coef", C.c_float), ("reward_coef", C.c_float),
        ("params", DynState), ("adam_m", DynState), ("adam_v", DynState),
        ("t_shared", C.c_int), ("t_action", C.c_int), ("lr", C.c_float), ("nsplit", C.c_int),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_longlong), ("scalars_out", C.c_void_p),
    ]


_lib = None


def lib():
    """Load the C-ABI library (built in-tree by build.py); raise loudly if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"mobody_b200: {LIB_PATH} is missing. Build it with `python __graft_entry__.py` "
                "(nvcc, sm_100a). There is no CPU / eager fallback.")
        L = C.CDLL(LIB_PATH)
        L.mobody_last_error.restype = C.c_char_p
        L.mobody_abi_version.restype = C.c_int
        L.mobody_compact_scratch_ints.restype = C.c_longlong
        L.mobody_compact_scratch_ints.argtypes = [C.c_longlong]
        L.mobody_row_width.argtypes = [C.c_int, C.c_int]
        L.mobody_step.argtypes = [C.POINTER(StepDesc), C.c_void_p]
        L.mobody_rollout_stats_doubles.restype = C.c_int
        L.mobody_peer_push.argtypes = [C.POINTER(PeerDesc), C.c_void_p, C.c_void_p, C.c_void_p]
        L.mobody_peer_slot_floats.restype = C.c_longlong
        L.mobody_peer_slot_floats.argtypes = [C.c_longlong, C.c_int]
        L.mobody_peer_buffer_bytes.restype = C.c_longlong
        L.mobody_peer_buffer_bytes.argtypes = [C.c_int, C.c_longlong, C.c_int]
        L.mobody_peer_header.argtypes = [C.POINTER(PeerDesc), C.c_void_p, C.c_void_p, C.c_void_p]
        L.mobody_peer_ack.argtypes = [C.POINTER(PeerDesc), C.c_uint, C.c_void_p]
        L.mobody_peer_wait.argtypes = [C.POINTER(PeerDesc), C.c_void_p]
        L.mobody_peer_slot.argtypes = [C.POINTER(PeerDesc), C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
        L.mobody_rollout.argtypes = [C.POINTER(RolloutDesc), C.c_void_p]
        L.mobody_model_eval_workspace_bytes.restype = C.c_longlong
        L.mobody_model_eval_workspace_bytes.argtypes = [C.c_int, C.c_int, C.c_int]
        L.mobody_model_eval.argtypes = [C.POINTER(ModelEvalDesc), C.c_void_p]
        L.mobody_policy_forward.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(MlpParams), C.c_float,
                                            C.c_void_p, C.c_void_p]
        L.mobody_termination.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.mobody_gather_rows.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p]
        L.mobody_philox_indices.argtypes = [C.c_void_p, C.c_longlong, C.c_ulonglong, C.c_uint, C.c_uint, C.c_void_p]
        L.mobody_sample_rows.argtypes = [C.POINTER(SampleJob), C.c_int, C.c_int, C.c_void_p]
        L.mobody_pack_rows.argtypes = [C.c_void_p] * 5 + [C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.mobody_ring_insert.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_int, C.c_longlong, C.c_longlong,
                                         C.c_void_p, C.c_void_p]
        L.mobody_ring_insert_transitions.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.c_longlong,
                                                     C.c_void_p, C.c_void_p]
        L.mobody_compact.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_longlong, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p]
        L.mobody_gather_pos.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p,
                                        C.c_int, C.c_void_p]
        L.mobody_gather_pos_i64.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]
        L.mobody_dyn_pack_bytes.restype = C.c_longlong
        L.mobody_dyn_pack_bytes.argtypes = [C.c_int, C.c_int, C.c_int]
        L.mobody_dyn_pack.argtypes = [C.POINTER(DynParams), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.mobody_mlp_pack_bytes.restype = C.c_longlong
        L.mobody_mlp_pack_bytes.argtypes = [C.c_int, C.c_int, C.c_int]
        L.mobody_mlp_pack.argtypes = [C.POINTER(MlpParams), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.mobody_par_penalty.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]
        L.mobody_train_workspace_bytes.restype = C.c_longlong
        L.mobody_train_workspace_bytes.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
        L.mobody_train_step.argtypes = [C.POINTER(TrainDesc), C.c_void_p]
        L.mobody_train_ex_workspace_bytes.restype = C.c_longlong
        L.mobody_train_ex_workspace_bytes.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
        L.mobody_train_step_ex.argtypes = [C.POINTER(TrainExDesc), C.c_void_p]
        L.mobody_classifier_workspace_bytes.restype = C.c_longlong
        L.mobody_classifier_workspace_bytes.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
        L.mobody_classifier_step.argtypes = [C.POINTER(ClassifierDesc), C.c_void_p]
        L.mobody_dara_relabel.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.POINTER(MlpParams),
                                          C.POINTER(MlpParams), C.c_float, C.c_void_p, C.c_void_p]
        L.mobody_dynfit_workspace_bytes.restype = C.c_longlong
        L.mobody_dynfit_workspace_bytes.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
        L.mobody_dynfit_step.argtypes = [C.POINTER(DynFitDesc), C.c_void_p]
        L.mobody_selftest_gemm.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.mobody_selftest_umma.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        if L.mobody_abi_version() != ABI_VERSION:
            raise RuntimeError("mobody_b200: ABI version mismatch between _ffi.py and libmobody_b200.so")
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise RuntimeError(f"mobody_b200 [{rc}]: {lib().mobody_last_error().decode()}")


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("mobody_b200: expected a CUDA tensor (there is no CPU path)")
    if not t.is_contiguous():
        raise RuntimeError("mobody_b200: expected a contiguous tensor")
    return t.data_ptr()


def f32(t, device):
    """Plumbing: make `t` a contiguous fp32 tensor on `device` (accepts numpy / CPU tensors)."""
    if not torch.is_tensor(t):
        t = torch.as_tensor(t)
    return t.to(device=device, dtype=torch.float32, non_blocking=True).contiguous()


def dyn_params(model):
    """DynParams of a MOBODYModule-like nn.Module (live parameter storage, no copies)."""
    d = DynParams()
    keep = []
    for i, name in enumerate(DYN_LAYER_NAMES):
        lay = getattr(model, name)
        w, b = lay.weight.detach(), lay.bias.detach()
        if w.dtype != torch.float32 or not w.is_cuda or not w.is_contiguous() or not b.is_contiguous():
            raise RuntimeError(f"mobody_b200: {name} parameters must be contiguous fp32 CUDA tensors")
        d.w[i], d.b[i] = w.data_ptr(), b.data_ptr()
        keep += [w, b]
    return d, keep


def mlp_state(tensors):
    """MlpState from [w0, b0, w1, b1, w2, b2] contiguous fp32 CUDA tensors (parameters or Adam moments)."""
    st = MlpState()
    for i in range(3):
        w, b = tensors[2 * i], tensors[2 * i + 1]
        if w.dtype != torch.float32 or not w.is_cuda or not w.is_contiguous() or not b.is_contiguous():
            raise RuntimeError("mobody_b200: train-step tensors must be contiguous fp32 CUDA tensors")
        st.w[i], st.b[i] = w.data_ptr(), b.data_ptr()
    return st


def mlp_tensors(mlp):
    """[w0, b0, w1, b1, w2, b2] parameter tensors (detached views of the live storage) of an MLPNetwork."""
    net = mlp.network
    return [t.detach() for li in (0, 2, 4) for t in (net[li].weight, net[li].bias)]


def mlp_params(mlp):
    """MlpParams of an MLPNetwork-like module with .network = Sequential(Linear,ReLU,Linear,ReLU,Linear)."""
    net = mlp.network
    m = MlpParams()
    keep = []
    for i, li in enumerate((0, 2, 4)):
        w, b = net[li].weight.detach(), net[li].bias.detach()
        if w.dtype != torch.float32 or not w.is_cuda or not w.is_contiguous():
            raise RuntimeError("mobody_b200: MLP parameters must be contiguous fp32 CUDA tensors")
        m.w[i], m.b[i] = w.data_ptr(), b.data_ptr()
        keep += [w, b]
    return m, keep
