"""ctypes binding of include/gcnbmp.h (the C-ABI of libgcnbmp.so).

This is the stub INTEGRATION.md shows a reference maintainer: structures mirror
the header field for field; device pointers are plain integers
(`torch.Tensor.data_ptr()` here, `cupy.ndarray.data.ptr` in a Chainer process).
There is no CPU fallback: if the library is missing this module raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgcnbmp.so")

MAX_STEPS = 16
OK, EINVAL, ESHAPE, EARCH, ECUDA = 0, -1, -2, -3, -4
ACT = {"identity": 0, "tanh": 1, "relu": 2, "sigmoid": 3}
READOUT_R1, READOUT_R2, READOUT_SUM = 1, 2, 3
COATTN_FINE, COATTN_POOL = 0, 1
PAIR_SYM, PAIR_PROD, PAIR_CONCAT = 0, 1, 2
MODE_F32, MODE_BF16 = 0, 1

fp = C.c_void_p   # device pointer
_A = lambda: fp * MAX_STEPS


class GRU(C.Structure):
    _fields_ = [(n, fp) for n in ("W_r", "b_Wr", "U_r", "b_Ur", "W_z", "b_Wz", "U_z", "b_Uz", "W", "b_W", "U", "b_U")]


class GgnnFwd(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("mb", "n_atoms", "hidden", "n_edge", "n_steps", "n_atom_types", "mode")] + [
        ("atoms", fp), ("h_in", fp), ("embed_W", fp), ("adj", fp), ("state_in", fp),
        ("msg_W", _A()), ("msg_b", _A()), ("gru", GRU * MAX_STEPS), ("stateful", C.c_int * MAX_STEPS),
        ("h_out", fp), ("h0_out", fp), ("Hs", fp), ("Ms", fp), ("Gs", fp), ("RSs", fp),
        ("tc_workspace", fp), ("tc_workspace_bytes", C.c_size_t), ("stash2", fp), ("tc_images_ready", C.c_int), ("adj_u8", C.c_int),
        ("mol_index", fp)]


class GgnnBwd(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("mb", "n_atoms", "hidden", "n_edge", "n_steps", "mode")] + [
        ("adj", fp), ("state_in", fp), ("msg_W", _A()), ("gru", GRU * MAX_STEPS),
        ("stateful", C.c_int * MAX_STEPS), ("Hs", fp), ("Ms", fp), ("RSs", fp), ("Gs", fp), ("Ps", fp), ("dHs", fp),
        ("d_msg_W", _A()), ("d_msg_b", _A()), ("d_gru", GRU * MAX_STEPS), ("d_state_in", fp),
        ("tc_workspace", fp), ("tc_workspace_bytes", C.c_size_t), ("stash2", fp), ("tc_images_ready", C.c_int), ("adj_u8", C.c_int),
        ("mol_index", fp), ("dHs_every_step", C.c_int), ("det_scratch", fp), ("det_scratch_bytes", C.c_size_t)]


class Pair(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("mb", "n1", "n2", "hidden", "out_dim", "head", "n_classes", "n_steps", "n_atom_types", "mode",
                                       "coattn_variant", "coattn_act")] + [
        ("atoms_1", fp), ("atoms_2", fp), ("adj_1", fp), ("adj_2", fp), ("labels", fp), ("count", C.c_float), ("embed_W", fp),
        ("msg_W", _A()), ("msg_b", _A()), ("gru", GRU * MAX_STEPS), ("stateful", C.c_int * MAX_STEPS)] + [
        (n, fp) for n in ("W", "V1", "V2", "b", "lt_1", "lt_2", "wa_1", "wa_2", "W_j", "b_j", "out_W", "out_b", "d_embed_W")] + [
        ("d_msg_W", _A()), ("d_msg_b", _A()), ("d_gru", GRU * MAX_STEPS)] + [
        (n, fp) for n in ("d_W", "d_V1", "d_V2", "d_b", "d_lt_1", "d_lt_2", "d_wa_1", "d_wa_2", "d_W_j", "d_b_j", "d_out_W", "d_out_b",
                          "logits", "loss", "workspace")] + [("workspace_bytes", C.c_size_t), ("adj_u8", C.c_int)]


class Bimpm(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("mb", "n1", "n2", "hidden", "head")] + [
        ("atoms_1", fp), ("atoms_2", fp), ("max_pooling_W", fp), ("att_mean_W", fp), ("att_max_W", fp),
        ("out_1", fp), ("out_2", fp), ("d_out_1", fp), ("d_out_2", fp), ("d_atoms_1", fp), ("d_atoms_2", fp),
        ("d_max_pooling_W", fp), ("d_att_mean_W", fp), ("d_att_max_W", fp), ("workspace", fp), ("workspace_bytes", C.c_size_t)]


class RelgcnFwd(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("mb", "n_atoms", "n_edge", "n_layers", "n_atom_types", "scale_adj", "act")] + [
        ("ch", C.c_int * (MAX_STEPS + 1)), ("atoms", fp), ("h_in", fp), ("embed_W", fp), ("adj", fp),
        ("self_W", _A()), ("self_b", _A()), ("edge_W", _A()), ("edge_b", _A()), ("h_out", fp), ("Hs", fp),
        ("mode", C.c_int), ("tc_workspace", fp), ("tc_workspace_bytes", C.c_size_t), ("stash2", fp), ("tc_images_ready", C.c_int), ("adj_u8", C.c_int)]


class RelgcnBwd(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("mb", "n_atoms", "n_edge", "n_layers", "scale_adj", "act")] + [
        ("ch", C.c_int * (MAX_STEPS + 1)), ("adj", fp), ("self_W", _A()), ("edge_W", _A()), ("Hs", fp),
        ("d_h_out", fp), ("Ds", fp), ("Ps", fp), ("d_h0", fp),
        ("d_self_W", _A()), ("d_self_b", _A()), ("d_edge_W", _A()), ("d_edge_b", _A()),
        ("mode", C.c_int), ("tc_workspace", fp), ("tc_workspace_bytes", C.c_size_t), ("stash2", fp), ("tc_images_ready", C.c_int), ("adj_u8", C.c_int), ("det_scratch", fp), ("det_scratch_bytes", C.c_size_t)]


class ReadoutFwd(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("mb", "n_atoms", "hidden", "out_dim", "variant", "act", "act_agg")] + [
        (n, fp) for n in ("h", "h0", "is_real_node", "W_i", "b_i", "W_j", "b_j", "g")] + [
        ("mode", C.c_int), ("tc_workspace", fp), ("tc_workspace_bytes", C.c_size_t), ("tc_images_ready", C.c_int)]


class ReadoutBwd(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("mb", "n_atoms", "hidden", "out_dim", "variant", "act", "act_agg")] + [
        (n, fp) for n in ("h", "h0", "is_real_node", "W_i", "b_i", "W_j", "b_j", "g", "dg",
                          "DU", "DV", "dh", "dh0", "d_W_i", "d_b_i", "d_W_j", "d_b_j")] + [
        ("mode", C.c_int), ("tc_workspace", fp), ("tc_workspace_bytes", C.c_size_t), ("tc_images_ready", C.c_int), ("det_scratch", fp), ("det_scratch_bytes", C.c_size_t)]


_CO_PARAMS = ("W", "V1", "V2", "b", "lt_1", "lt_2", "wa_1", "wa_2", "W_j", "b_j")


class CoattnFwd(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("mb", "n1", "n2", "hidden", "out_dim", "head", "variant", "act")] + [
        (n, fp) for n in ("atoms_1", "atoms_2") + _CO_PARAMS + ("compact_1", "compact_2")] + [
        ("mode", C.c_int), ("tc_workspace", fp), ("tc_workspace_bytes", C.c_size_t), ("tc_images_ready", C.c_int)]


class CoattnBwd(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("mb", "n1", "n2", "hidden", "out_dim", "head", "variant", "act")] + [
        (n, fp) for n in ("atoms_1", "atoms_2") + _CO_PARAMS + ("d_compact_1", "d_compact_2", "R", "P1", "P2",
                                                             "DL1", "DL2", "d_atoms_1", "d_atoms_2")
        + tuple("d_" + p for p in _CO_PARAMS)] + [
        ("mode", C.c_int), ("tc_workspace", fp), ("tc_workspace_bytes", C.c_size_t), ("tc_images_ready", C.c_int), ("det_scratch", fp), ("det_scratch_bytes", C.c_size_t)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "gcnbmp: %s is missing -- build it with `python gcn-bmp_b200/build.py` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    i, i64, f, vp = C.c_int, C.c_int64, C.c_float, C.c_void_p
    sig = {
        "bmp_ggnn_forward": [C.POINTER(GgnnFwd), vp],
        "bmp_ggnn_backward": [C.POINTER(GgnnBwd), vp],
        "bmp_embed_backward": [fp, fp, fp, i, i, i, vp],
        "bmp_relgcn_forward": [C.POINTER(RelgcnFwd), vp],
        "bmp_relgcn_backward": [C.POINTER(RelgcnBwd), vp],
        "bmp_rescale_adj": [fp, fp, i, i, i, vp],
        "bmp_readout_forward": [C.POINTER(ReadoutFwd), vp],
        "bmp_readout_backward": [C.POINTER(ReadoutBwd), vp],
        "bmp_coattn_forward": [C.POINTER(CoattnFwd), vp],
        "bmp_coattn_backward": [C.POINTER(CoattnBwd), vp],
        "bmp_hole_corr_forward": [fp, fp, fp, i, i, vp],
        "bmp_hole_corr_backward": [fp, fp, fp, fp, fp, i, i, vp],
        "bmp_linear_forward": [fp, fp, fp, fp, i, i, i, i, vp],
        "bmp_linear_backward": [fp, fp, fp, fp, fp, fp, fp, i, i, i, i, vp],
        "bmp_wgrad": [fp, i, fp, i, fp, i, i64, i, i, vp],
        "bmp_wgrad_tc": [fp, i, fp, i, fp, i, i64, i, i, fp, i, vp],
        "bmp_wgrad_tc3": [fp, i, fp, i, fp, i, i64, i, i, fp, i, vp],
        "bmp_colsum": [fp, i, fp, i, i64, i, vp],
        "bmp_sigmoid_ce": [fp, fp, fp, fp, i, f, vp],
        "bmp_adam_step": [fp, fp, fp, fp, i, f, f, f, f, f, i, vp],
        "bmp_pair_features_forward": [fp, fp, fp, i, i, i, vp],
        "bmp_pair_features_backward": [fp, fp, fp, fp, fp, i, i, i, vp],
        "bmp_bilinear_forward": [fp, fp, fp, fp, fp, fp, fp, fp, i, i, i, i, vp],
        "bmp_bilinear_backward": [fp] * 14 + [i, i, i, i, vp],
        "bmp_grad_hooks": [fp, fp, i, f, f, f, fp, vp],
        "bmp_atoms_bcast_add_act_forward": [fp, fp, fp, i, i, i, i, vp],
        "bmp_atoms_bcast_add_act_backward": [fp, fp, fp, fp, i, i, i, i, vp],
        "bmp_atoms_softmax_forward": [fp, fp, i, i, i, vp],
        "bmp_atoms_softmax_backward": [fp, fp, fp, i, i, i, vp],
        "bmp_atoms_pool_forward": [fp, i, fp, fp, i, i, i, vp],
        "bmp_atoms_pool_backward": [fp, i, fp, fp, fp, fp, i, i, i, vp],
        "bmp_gin_aggregate": [fp, fp, fp, i, i, i, i, i, vp],
        "bmp_nfp_gather": [fp, fp, fp, i, i, i, i, i, vp],
        "bmp_bimpm_forward": [C.POINTER(Bimpm), vp],
        "bmp_bimpm_backward": [C.POINTER(Bimpm), vp],
        "bmp_embed_forward": [fp, fp, fp, i, i, i, vp],
        "bmp_linear_backward_det": [fp, fp, fp, fp, fp, fp, fp, i, i, i, i, vp, vp, C.c_size_t],
        "bmp_embed_backward_det": [fp, fp, fp, i, i, i, vp, vp, C.c_size_t],
        "bmp_sigmoid_ce_det": [fp, fp, fp, fp, i, f, vp, vp, C.c_size_t],
        "bmp_grad_hooks_det": [fp, fp, i, f, f, f, fp, vp, vp, C.c_size_t],
        "bmp_bilinear_backward_det": [fp] * 14 + [i, i, i, i, vp, vp, C.c_size_t],
    }
    for name, args in sig.items():
        fn = getattr(lib, name)
        fn.argtypes, fn.restype = args, C.c_int
    lib.bmp_ggnn_tc_workspace_bytes.argtypes, lib.bmp_ggnn_tc_workspace_bytes.restype = [i, i], C.c_size_t
    lib.bmp_ggnn_stash2_bytes.argtypes, lib.bmp_ggnn_stash2_bytes.restype = [i, i, i], C.c_size_t
    lib.bmp_ggnn_x3_workspace_bytes.argtypes, lib.bmp_ggnn_x3_workspace_bytes.restype = [i, i, i, i, i, i], C.c_size_t
    lib.bmp_ggnn_x3_forward_bytes.argtypes, lib.bmp_ggnn_x3_forward_bytes.restype = [C.c_void_p, i], C.c_size_t
    lib.bmp_pair_workspace_bytes.argtypes, lib.bmp_pair_workspace_bytes.restype = [i] * 9, C.c_size_t
    lib.bmp_pair_forward_backward.argtypes, lib.bmp_pair_forward_backward.restype = [C.c_void_p, vp], C.c_int
    lib.bmp_readout_tc_workspace_bytes.argtypes, lib.bmp_readout_tc_workspace_bytes.restype = [i, i], C.c_size_t
    lib.bmp_readout_x3_workspace_bytes.argtypes, lib.bmp_readout_x3_workspace_bytes.restype = [i] * 6, C.c_size_t
    lib.bmp_coattn_tc_workspace_bytes.argtypes, lib.bmp_coattn_tc_workspace_bytes.restype = [i], C.c_size_t
    lib.bmp_coattn_large_workspace_bytes.argtypes, lib.bmp_coattn_large_workspace_bytes.restype = [i] * 4, C.c_size_t
    lib.bmp_relgcn_tc_workspace_bytes.argtypes, lib.bmp_relgcn_tc_workspace_bytes.restype = [i, i], C.c_size_t
    lib.bmp_relgcn_x3_workspace_bytes.argtypes, lib.bmp_relgcn_x3_workspace_bytes.restype = [i] * 5, C.c_size_t
    lib.bmp_bimpm_workspace_bytes.argtypes, lib.bmp_bimpm_workspace_bytes.restype = [i, i, i, i, i], C.c_size_t
    for name in ("bmp_ggnn_backward_det_bytes", "bmp_relgcn_backward_det_bytes", "bmp_readout_backward_det_bytes",
                 "bmp_coattn_backward_det_bytes"):
        getattr(lib, name).argtypes, getattr(lib, name).restype = [C.c_void_p], C.c_size_t
    lib.bmp_linear_backward_det_bytes.argtypes, lib.bmp_linear_backward_det_bytes.restype = [i, i, i], C.c_size_t
    lib.bmp_embed_backward_det_bytes.argtypes, lib.bmp_embed_backward_det_bytes.restype = [i, i, i], C.c_size_t
    lib.bmp_sigmoid_ce_det_bytes.argtypes, lib.bmp_sigmoid_ce_det_bytes.restype = [i], C.c_size_t
    lib.bmp_grad_hooks_det_bytes.argtypes, lib.bmp_grad_hooks_det_bytes.restype = [i], C.c_size_t
    lib.bmp_bilinear_backward_det_bytes.argtypes, lib.bmp_bilinear_backward_det_bytes.restype = [i, i, i, i], C.c_size_t
    lib.bmp_last_error.restype = C.c_char_p
    lib.bmp_version.restype = C.c_int
    lib.bmp_device_check.restype = C.c_int
    lib.bmp_launch_count.restype = C.c_uint64
    lib.bmp_reset_launch_count.restype = None
    lib.bmp_profile_enable.argtypes, lib.bmp_profile_enable.restype = [i], None
    lib.bmp_profile_read.argtypes, lib.bmp_profile_read.restype = [C.POINTER(C.c_double), C.POINTER(C.c_longlong), i], C.c_int
    return lib


lib = _load()
EXPORTS = ["bmp_ggnn_forward", "bmp_ggnn_backward", "bmp_embed_backward", "bmp_relgcn_forward",
           "bmp_relgcn_backward", "bmp_relgcn_tc_workspace_bytes", "bmp_relgcn_x3_workspace_bytes", "bmp_rescale_adj", "bmp_readout_forward", "bmp_readout_backward", "bmp_readout_tc_workspace_bytes", "bmp_coattn_forward",
           "bmp_coattn_backward", "bmp_coattn_tc_workspace_bytes", "bmp_coattn_large_workspace_bytes", "bmp_hole_corr_forward", "bmp_hole_corr_backward", "bmp_linear_forward",
           "bmp_linear_backward", "bmp_ggnn_tc_workspace_bytes", "bmp_ggnn_stash2_bytes", "bmp_ggnn_x3_workspace_bytes", "bmp_ggnn_x3_forward_bytes", "bmp_pair_workspace_bytes", "bmp_pair_forward_backward", "bmp_readout_x3_workspace_bytes", "bmp_wgrad", "bmp_wgrad_tc", "bmp_wgrad_tc3", "bmp_colsum", "bmp_sigmoid_ce", "bmp_adam_step",
           "bmp_pair_features_forward", "bmp_pair_features_backward", "bmp_bilinear_forward", "bmp_bilinear_backward", "bmp_grad_hooks",
           "bmp_atoms_bcast_add_act_forward", "bmp_atoms_bcast_add_act_backward", "bmp_atoms_softmax_forward", "bmp_atoms_softmax_backward",
           "bmp_atoms_pool_forward", "bmp_atoms_pool_backward", "bmp_gin_aggregate", "bmp_nfp_gather", "bmp_embed_forward", "bmp_bimpm_forward", "bmp_bimpm_backward", "bmp_bimpm_workspace_bytes",
           "bmp_last_error", "bmp_version", "bmp_device_check", "bmp_launch_count", "bmp_reset_launch_count",
           "bmp_profile_enable", "bmp_profile_read",
           "bmp_ggnn_backward_det_bytes", "bmp_relgcn_backward_det_bytes", "bmp_readout_backward_det_bytes", "bmp_coattn_backward_det_bytes",
           "bmp_linear_backward_det", "bmp_linear_backward_det_bytes", "bmp_embed_backward_det", "bmp_embed_backward_det_bytes",
           "bmp_sigmoid_ce_det", "bmp_sigmoid_ce_det_bytes", "bmp_grad_hooks_det", "bmp_grad_hooks_det_bytes",
           "bmp_bilinear_backward_det", "bmp_bilinear_backward_det_bytes"]


class BmpError(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, "gcnbmp error %d: %s" % (code, msg))
        self.code = code


def check(rc):
    if rc != 0:
        msg = lib.bmp_last_error().decode("utf-8", "replace")
        if rc == ESHAPE:
            raise ValueError("gcnbmp: %s" % msg)
        raise BmpError(rc, msg)


def launch_count():
    return int(lib.bmp_launch_count())


def reset_launch_count():
    lib.bmp_reset_launch_count()


PROF_KINDS = ("ggnn_fwd", "ggnn_bwd", "wgrad", "coattn_fwd", "coattn_bwd", "readout")


def profile_enable(on=True):
    """CUDA events around every launch of the hot tcgen05 kernels, on the launching stream (include/gcnbmp.h)."""
    lib.bmp_profile_enable(1 if on else 0)


def profile_read():
    """-> {kind: (total ms, launches)} since the last read (synchronises on the recorded events)."""
    n = len(PROF_KINDS)
    ms, cnt = (C.c_double * n)(), (C.c_longlong * n)()
    check(lib.bmp_profile_read(ms, cnt, n))
    return {k: (float(ms[j]), int(cnt[j])) for j, k in enumerate(PROF_KINDS)}
