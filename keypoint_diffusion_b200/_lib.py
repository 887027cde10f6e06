"""ctypes binding of libkpdiff_b200.so (the C ABI declared in include/kpdiff_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C keypoint_diffusion_b200/csrc``.
There is no CPU fallback: if the shared library is missing, importing this module raises.
"""
import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ["KPD_LIB"]) if os.environ.get("KPD_LIB") else _HERE / "libkpdiff_b200.so"   # KPD_LIB: an instrumented build (tools/)

TILE_EDGES = 64


class KpdBatch(C.Structure):
    _fields_ = [("B", C.c_int32), ("n_lig", C.c_int32), ("n_kp", C.c_int32), ("max_lig", C.c_int32),
                ("max_kp", C.c_int32), ("lig_ptr", C.c_void_p), ("kp_ptr", C.c_void_p),
                ("lig_batch", C.c_void_p), ("kp_batch", C.c_void_p)]


class KpdCsr(C.Structure):
    _fields_ = [("n_dst", C.c_int32), ("cap", C.c_int32), ("rowptr", C.c_void_p), ("src", C.c_void_p),
                ("dst", C.c_void_p)]


class KpdGraphParams(C.Structure):
    _fields_ = [("ll_k", C.c_int32), ("ll_cap", C.c_int32), ("kl_k", C.c_int32), ("kl_cap", C.c_int32),
                ("ll_r", C.c_double), ("kl_r", C.c_double)]


class KpdEgnnConfig(C.Structure):
    _fields_ = [("atom_nf", C.c_int32), ("rec_nf", C.c_int32), ("hidden_nf", C.c_int32), ("n_layers", C.c_int32),
                ("use_tanh", C.c_int32), ("update_kp_feat", C.c_int32), ("norm", C.c_int32),
                ("has_rec_encoder", C.c_int32), ("coords_range", C.c_float), ("message_norm", C.c_float),
                ("z_effective", C.c_int32)]


class KpdGvpConfig(C.Structure):
    _fields_ = [("n_lig_scalars", C.c_int32), ("n_kp_scalars", C.c_int32), ("vector_size", C.c_int32),
                ("n_convs", C.c_int32), ("n_hidden_scalars", C.c_int32), ("n_message_gvps", C.c_int32),
                ("n_update_gvps", C.c_int32), ("n_noise_gvps", C.c_int32), ("update_kp", C.c_int32),
                ("norm_mode", C.c_int32), ("message_norm", C.c_float), ("rbf_dmax", C.c_float),
                ("rbf_dim", C.c_int32)]


class KpdSamplerConfig(C.Structure):
    _fields_ = [("arch", C.c_int32), ("T", C.c_int32), ("atom_nf", C.c_int32), ("steps_per_graph", C.c_int32),
                ("use_cuda_graph", C.c_int32), ("lig_feat_norm_constant", C.c_float)]


def _load():
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} not found: the CUDA library is the only implementation of this path "
            "(no CPU fallback). Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C keypoint_diffusion_b200/csrc`.")
    lib = C.CDLL(str(LIB_PATH), mode=os.RTLD_LOCAL)
    P, I, L, F, U64 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_uint64
    sig = {
        "kpd_last_error": (C.c_char_p, []),
        "kpd_version": (I, []),
        "kpd_launch_count": (L, []),
        "kpd_profile_enable": (I, [I, I]),
        "kpd_profile_collect": (I, [C.POINTER(C.c_double), C.POINTER(I)]),
        "kpd_sampler_edge_stats": (I, [P, C.POINTER(C.c_double)]),
        "kpd_graph_workspace_bytes": (L, [C.POINTER(KpdBatch)]),
        "kpd_build_graph": (I, [C.POINTER(KpdBatch), P, P, C.POINTER(KpdGraphParams), C.POINTER(KpdCsr),
                                C.POINTER(KpdCsr), C.POINTER(KpdCsr), P, P, P, P]),
        "kpd_linear": (I, [P, I, P, I, P, P, I, P, I, I, I, I, I, P]),
        "kpd_tc_linear": (I, [P, I, P, P, P, I, P, I, I, I, I, I, I, P]),
        "kpd_egnn_create": (I, [C.POINTER(KpdEgnnConfig), P, C.POINTER(L), I, C.POINTER(P)]),
        "kpd_egnn_destroy": (None, [P]),
        "kpd_egnn_attach_tc": (I, [P, P, C.POINTER(L), I, I]),
        "kpd_egnn_set_mode": (I, [P, I]),
        "kpd_debug_ws_times": (I, [P]),
        "kpd_debug_eg_times": (I, [P]),
        "kpd_debug_ws_trace": (I, [P, I, P]),
        "kpd_debug_timeline": (I, [P, I]),
        "kpd_egnn_dims": (I, [P, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
        "kpd_egnn_workspace_bytes": (L, [P, C.POINTER(KpdBatch), I, I, I]),
        "kpd_egnn_forward": (I, [P, C.POINTER(KpdBatch), P, P, P, P, P, P, I, C.POINTER(KpdCsr),
                                 C.POINTER(KpdCsr), C.POINTER(KpdCsr), C.POINTER(KpdCsr), P, P, P, P]),
        "kpd_egnn_encode_kp": (I, [P, P, I, P, P, P]),
        "kpd_gvp_create": (I, [C.POINTER(KpdGvpConfig), P, C.POINTER(L), I, C.POINTER(P)]),
        "kpd_gvp_destroy": (None, [P]),
        "kpd_gvp_attach_tc": (I, [P, P, C.POINTER(L), I, I]),
        "kpd_gvp_set_mode": (I, [P, I]),
        "kpd_gvp_dims": (I, [P, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
        "kpd_gvp_workspace_bytes": (L, [P, C.POINTER(KpdBatch), I, I, I]),
        "kpd_gvp_forward": (I, [P, C.POINTER(KpdBatch), P, P, P, P, P, P, I, C.POINTER(KpdCsr),
                                C.POINTER(KpdCsr), C.POINTER(KpdCsr), C.POINTER(KpdCsr), P, P, P, P]),
        "kpd_ddpm_step": (I, [C.POINTER(KpdBatch), P, P, P, P, P, I, P, P, P, P, U64, P]),
        "kpd_ddpm_multistep_step": (I, [C.POINTER(KpdBatch), P, P, P, P, P, I, P, P, P, I, P, P, P, P, U64, P]),
        "kpd_ddpm_inpaint_step": (I, [C.POINTER(KpdBatch), P, P, P, P, P, I, P, P, P, I, P, P, P, P, F, P, U64, P]),
        "kpd_renoise": (I, [C.POINTER(KpdBatch), P, P, P, I, P, P, I, P, U64, P]),
        "kpd_remove_com": (I, [C.POINTER(KpdBatch), P, P, I, P, P]),
        "kpd_shift_by_complex": (I, [P, P, I, P, F, P]),
        "kpd_randn_init": (I, [P, P, I, I, U64, P]),
        "kpd_sampler_create": (I, [C.POINTER(KpdSamplerConfig), P, C.POINTER(KpdBatch), C.POINTER(KpdGraphParams),
                                   C.POINTER(KpdCsr), I, P, I, I, P, L, C.POINTER(P)]),
        "kpd_sampler_workspace_bytes": (L, [C.POINTER(KpdSamplerConfig), P, C.POINTER(KpdBatch), I, I, I]),
        "kpd_sampler_destroy": (None, [P]),
        "kpd_sampler_run": (I, [P, P, P, P, P, P, P, P, U64, I, P]),
        "kpd_sampler_launches_per_step": (I, [P]),
        "kpd_sampler_set_atom_offset": (I, [P, I]),
        "kpd_sampler_enable_inpainting": (I, [P, I, P]),
        "kpd_sampler_set_fragment": (I, [P, P, P, P]),
        "kpd_sampler_set_start": (I, [P, I, P, P, F, F]),
        "kpd_sampler_set_schedule": (I, [P, I, P, P]),
        "kpd_sampler_enable_recording": (I, [P]),
        "kpd_sampler_set_recording": (I, [P, I, I, P, P, P, P, I, P]),
        "kpd_sampler_enable_multistep": (I, [P]),
        "kpd_sampler_set_multistep": (I, [P, I, P, P, P]),
        "kpd_partial_noise": (I, [C.POINTER(KpdBatch), P, P, P, P, P, I, F, F, F, P, U64, P]),
        "kpd_decode_atom_types": (I, [P, I, I, P, P]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib, sorted(sig)


lib, EXPORTED = _load()


def check(rc, what=""):
    if rc != 0:
        msg = lib.kpd_last_error()
        raise RuntimeError(f"kpdiff_b200 {what} failed ({rc}): {msg.decode() if msg else ''}")


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())
