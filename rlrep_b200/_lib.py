"""ctypes binding of librlrep_b200.so (C ABI declared in include/rlrep_b200.h).

There is exactly one compute path: the CUDA library.  If the shared object is missing or a call fails the
caller gets an exception -- nothing here falls back to PyTorch or to the CPU oracle.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "librlrep_b200.so"


class RlrepError(RuntimeError):
    pass


class OptimState(C.Structure):
    """Mirror of `rlrep_optim_state` (include/rlrep_b200.h)."""
    _fields_ = [("steps", C.c_int), ("t_feature", C.c_longlong), ("t_critic", C.c_longlong), ("t_actor", C.c_longlong),
                ("t_alpha", C.c_longlong), ("log_alpha", C.c_double), ("log_alpha_m", C.c_double),
                ("log_alpha_v", C.c_double)]


class AgentConfig(C.Structure):
    """Mirror of `rlrep_agent_config` (include/rlrep_b200.h)."""
    _fields_ = [
        ("alg", C.c_int), ("state_dim", C.c_int), ("action_dim", C.c_int), ("batch_size", C.c_int),
        ("hidden_dim", C.c_int), ("feature_dim", C.c_int), ("actor_hidden_dim", C.c_int), ("feature_steps", C.c_int),
        ("lr_critic", C.c_double), ("lr_feature", C.c_double), ("lr_actor", C.c_double), ("lr_alpha", C.c_double),
        ("discount", C.c_float), ("tau", C.c_float), ("feature_tau", C.c_float), ("alpha", C.c_double),
        ("target_update_period", C.c_int), ("auto_entropy_tuning", C.c_int), ("use_feature_target", C.c_int),
        ("precision", C.c_int), ("use_cuda_graph", C.c_int),
        ("phi_hidden_dim", C.c_int), ("phi_hidden_depth", C.c_int), ("mu_hidden_dim", C.c_int),
        ("mu_hidden_depth", C.c_int), ("nabla_mu_hidden_dim", C.c_int), ("nabla_mu_hidden_depth", C.c_int),
        ("num_noise", C.c_int), ("num_noises", C.c_int), ("sigma_scale_factor", C.c_float),
    ]


ALG = {"sac": 0, "ctrlsac": 1, "vlsac": 2, "spedersac": 3, "diffsrsac": 4}
PRECISION = {"tf32": 0, "fp32": 1}


class Epilogue(C.Structure):
    """Mirror of `rlrep_epilogue` (include/rlrep_b200.h)."""
    _fields_ = [
        ("bias", C.c_void_p), ("r1_u", C.c_void_p), ("r1_v", C.c_void_p), ("aux", C.c_void_p),
        ("pre_out", C.c_void_p), ("ld_aux", C.c_int), ("ld_pre", C.c_int), ("act", C.c_int),
        ("dact", C.c_int), ("accumulate", C.c_int), ("scale", C.c_float),
    ]


ACT = {"none": 0, "elu": 1, "relu": 2, "tanh": 3, "sin": 4}
DACT = {"none": 0, "elu_out": 1, "relu_out": 2, "tanh_out": 3, "cos_pre": 4}

_lib = None


def load() -> C.CDLL:
    """Load the library once.  Raises if it has not been built (python -m rlrep_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RlrepError(
            f"{LIB_PATH} not found: build it with `python -m rlrep_b200.build` (needs nvcc). "
            "rlrep_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(str(LIB_PATH))
    lib.rlrep_last_error.restype = C.c_char_p
    lib.rlrep_abi_version.restype = C.c_int
    _declare(lib)
    _lib = lib
    return lib


def _declare(lib: C.CDLL) -> None:
    vp, i, f, sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t
    sigs = {
        "rlrep_gemm": [vp, i, i, i, i, vp, i, i, vp, i, i, vp, i, i, vp, i, C.POINTER(Epilogue), i, i, vp, sz],
        "rlrep_gemm_bench": [vp, i, i, i, i, vp, i, i, vp, i, i, vp, i, C.POINTER(Epilogue), i, i, vp, sz, i,
                             C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_int)],
        "rlrep_gemm_trace": [vp],
        "rlrep_gemm_chain_begin": [],
        "rlrep_gemm_chain_set_debug": [vp],
        "rlrep_gemm_chain_add": [i, i, i, vp, i, i, vp, i, i, vp, i, C.POINTER(Epilogue)],
        "rlrep_gemm_chain_run": [vp, i, i, i, C.POINTER(C.c_float), C.POINTER(C.c_int)],
        "rlrep_ring_create": [i, i, C.c_longlong, C.POINTER(vp)],
        "rlrep_ring_destroy": [vp],
        "rlrep_ring_layout": [vp] + [C.POINTER(i)] * 5,
        "rlrep_ring_state": [vp] + [C.POINTER(C.c_longlong)] * 3,
        "rlrep_ring_add_packed": [vp, vp, i, vp],
        "rlrep_ring_load": [vp, vp, vp, vp, vp, vp, C.c_longlong, i, vp],
        "rlrep_ring_gather": [vp, vp, i, vp, vp],
        "rlrep_agent_create": [C.POINTER(AgentConfig), vp, C.POINTER(vp)],
        "rlrep_agent_destroy": [vp],
        "rlrep_conv_encoder_create": [i, i, i, i, vp, C.POINTER(vp)],
        "rlrep_conv_encoder_destroy": [vp],
        "rlrep_conv_encoder_read": [vp, i, i, vp],
        "rlrep_conv_encoder_write": [vp, i, i, vp],
        "rlrep_conv_encoder_forward": [vp, vp, vp, vp],
        "rlrep_conv_encoder_backward": [vp, vp],
        "rlrep_conv_encoder_feature_dim": [vp, C.POINTER(i)],
        "rlrep_conv_encoder_forward_pitched": [vp, vp, vp, vp, i, i],
        "rlrep_conv_encoder_backward_pitched": [vp, vp, i],
        "rlrep_conv_encoder_read_map": [vp, i, i, vp],
        "rlrep_conv_decoder_create": [i, i, i, vp, C.POINTER(vp)],
        "rlrep_conv_decoder_destroy": [vp],
        "rlrep_conv_decoder_read": [vp, i, i, vp],
        "rlrep_conv_decoder_write": [vp, i, i, vp],
        "rlrep_conv_decoder_forward": [vp, vp, i],
        "rlrep_conv_decoder_l1_loss": [vp, vp, f, vp],
        "rlrep_conv_decoder_mse_sum_loss": [vp, vp, vp, f, vp],
        "rlrep_conv_decoder_backward": [vp, vp, i],
        "rlrep_conv_decoder_read_map": [vp, i, i, vp],
        "rlrep_drq_create": [vp, vp, C.POINTER(vp)],
        "rlrep_drq_update": [vp, vp, vp, vp, vp, vp, vp, vp, C.c_float, vp],
        "rlrep_drq_act": [vp, vp, vp, C.c_float, vp],
        "rlrep_drq_act_batch": [vp, vp, vp, C.c_float, i, vp],
        "rlrep_gemm_set_debug_buffer": [vp],
        "rlrep_ldiff_create": [vp, vp, C.POINTER(vp)],
        "rlrep_ldiff_update": [vp, vp, vp],
        "rlrep_mulv_create": [vp, vp, C.POINTER(vp)],
        "rlrep_mulv_update": [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_float, vp],
        "rlrep_mulv_act": [vp, vp, vp, C.c_float, vp],
        "rlrep_mulv_act_batch": [vp, vp, vp, C.c_float, i, vp],
        "rlrep_comm_unique_id": [vp],
        "rlrep_comm_create": [vp, i, i, C.POINTER(vp)],
        "rlrep_comm_destroy": [vp],
        "rlrep_comm_info": [vp, C.POINTER(i), C.POINTER(i), C.POINTER(i), C.POINTER(C.c_longlong)],
        "rlrep_agent_create_sharded": [C.POINTER(AgentConfig), vp, vp, C.POINTER(vp)],
        "rlrep_agent_num_tensors": [vp, C.POINTER(i)],
        "rlrep_agent_tensor_info": [vp, i, C.POINTER(C.c_char_p), C.POINTER(vp), C.POINTER(i), C.POINTER(i)],
        "rlrep_agent_tensor_read": [vp, i, vp],
        "rlrep_agent_tensor_write": [vp, i, vp],
        "rlrep_agent_sync_targets": [vp],
        "rlrep_agent_get_log_alpha": [vp, C.POINTER(C.c_double)],
        "rlrep_agent_set_log_alpha": [vp, C.c_double],
        "rlrep_agent_get_steps": [vp, C.POINTER(i)],
        "rlrep_agent_get_optim_state": [vp, C.POINTER(OptimState)],
        "rlrep_agent_set_optim_state": [vp, C.POINTER(OptimState)],
        "rlrep_agent_train_counts": [vp, C.POINTER(i), C.POINTER(i), C.POINTER(i)],
        "rlrep_agent_train": [vp, vp, vp, i, vp, i, vp, i],
        "rlrep_agent_act": [vp, vp, vp, vp],
        "rlrep_pixring_create": [C.c_longlong, i, i, i, i, C.POINTER(vp)],
        "rlrep_pixring_destroy": [vp],
        "rlrep_pixring_write": [vp, C.c_longlong, i, vp, vp, C.c_float, C.c_float, i],
        "rlrep_pixring_flush": [vp],
        "rlrep_pixring_gather": [vp, vp, i, vp, C.c_float, vp, vp, vp, vp, vp, vp],
        "rlrep_agent_act_batch": [vp, vp, vp, i, vp],
        "rlrep_agent_last_launches": [vp, C.POINTER(i)],
        "rlrep_agent_graph_stats": [vp, C.POINTER(i), C.POINTER(i)],
        "rlrep_agent_train_resident": [vp, vp, vp, vp, i, C.POINTER(C.c_float)],
        "rlrep_agent_profile_train": [vp, vp, vp, vp, i, C.POINTER(C.c_char_p), C.POINTER(C.c_float),
                                      C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(i)],
    }
    # the pixel agents' handle entry points, the same for each agent (rlrep_drq_*, rlrep_mulv_*, rlrep_ldiff_*)
    for prefix in ("drq", "mulv", "ldiff"):
        sigs.update({
            f"rlrep_{prefix}_destroy": [vp],
            f"rlrep_{prefix}_num_tensors": [vp, C.POINTER(i)],
            f"rlrep_{prefix}_tensor_info": [vp, i, C.POINTER(C.c_char_p), C.POINTER(vp), C.POINTER(i), C.POINTER(i)],
            f"rlrep_{prefix}_tensor_read": [vp, i, vp],
            f"rlrep_{prefix}_tensor_write": [vp, i, vp],
            f"rlrep_{prefix}_sync_targets": [vp],
            f"rlrep_{prefix}_update_resident": [vp, i, C.c_float, C.POINTER(C.c_float)],
            f"rlrep_{prefix}_profile_update": [vp, C.c_float, i, C.POINTER(C.c_char_p), C.POINTER(C.c_float),
                                               C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(i)],
            f"rlrep_{prefix}_last_launches": [vp, C.POINTER(i)],
            f"rlrep_{prefix}_get_optim_state": [vp, C.POINTER(OptimState)],
            f"rlrep_{prefix}_set_optim_state": [vp, C.POINTER(OptimState)],
        })
    lib.rlrep_agent_metric_name.argtypes = [vp, i]
    lib.rlrep_agent_metric_name.restype = C.c_char_p
    for name, argtypes in sigs.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int


def check(rc: int) -> None:
    if rc != 0:
        msg = load().rlrep_last_error()
        raise RlrepError(msg.decode() if msg else f"rlrep call failed with code {rc}")


def current_stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


def make_epilogue(bias=None, r1=None, aux=None, pre_out=None, act="none", dact="none", accumulate=False,
                  scale=1.0) -> Epilogue:
    e = Epilogue()
    e.bias = bias.data_ptr() if bias is not None else None
    if r1 is not None:
        e.r1_u, e.r1_v = r1[0].data_ptr(), r1[1].data_ptr()
    if aux is not None:
        e.aux, e.ld_aux = aux.data_ptr(), aux.stride(0)
    if pre_out is not None:
        e.pre_out, e.ld_pre = pre_out.data_ptr(), pre_out.stride(0)
    e.act, e.dact = ACT[act], DACT[dact]
    e.accumulate = int(accumulate)
    e.scale = scale
    return e


def gemm(A, B, C_out, *, a_mn=False, b_mn=False, path="tc", epi: Epilogue | None = None, A2=None, bn=0, split_k=0,
         ws=None):
    """C = epilogue(sum_k A(m,k) B(n,k)) on torch CUDA tensors (kernel-level entry, used by tests).

    K-major operand: tensor [rows, K]; MN-major operand: tensor [K, rows]."""
    lib = load()
    M = A.shape[1] if a_mn else A.shape[0]
    K = A.shape[0] if a_mn else A.shape[1]
    N = B.shape[1] if b_mn else B.shape[0]
    K1 = K
    if A2 is not None:
        K += A2.shape[1]
    assert (B.shape[0] if b_mn else B.shape[1]) == K
    epi = epi or make_epilogue()
    rc = lib.rlrep_gemm(current_stream_ptr(), 0 if path == "tc" else 1, M, N, K, A.data_ptr(), A.stride(0), int(a_mn),
                        A2.data_ptr() if A2 is not None else None, A2.stride(0) if A2 is not None else 0, K1,
                        B.data_ptr(), B.stride(0), int(b_mn), C_out.data_ptr(), C_out.stride(0), C.byref(epi), bn,
                        split_k, ws.data_ptr() if ws is not None else None, ws.numel() if ws is not None else 0)
    check(rc)
    return C_out


def gemm_chain(specs, *, bn=0, split_k=0, iters=1):
    """Runs a DAG of GEMMs as ONE persistent chain kernel (csrc/gemm_chain.cuh).  specs = [(A, B, C_out, dict(a_mn=, b_mn=,
    epi=))] in program order; dependencies are inferred from the tensors' addresses.  Returns (ms per launch, levels)."""
    lib = load()
    check(lib.rlrep_gemm_chain_begin())
    keep = []
    for A, B, C_out, kw in specs:
        a_mn, b_mn = bool(kw.get("a_mn", False)), bool(kw.get("b_mn", False))
        M = A.shape[1] if a_mn else A.shape[0]
        K = A.shape[0] if a_mn else A.shape[1]
        N = B.shape[1] if b_mn else B.shape[0]
        assert (B.shape[0] if b_mn else B.shape[1]) == K
        epi = kw.get("epi") or make_epilogue()
        keep.append(epi)
        check(lib.rlrep_gemm_chain_add(M, N, K, A.data_ptr(), A.stride(0), int(a_mn), B.data_ptr(), B.stride(0), int(b_mn),
                                       C_out.data_ptr(), C_out.stride(0), C.byref(epi)))
    ms, levels = C.c_float(), C.c_int()
    check(lib.rlrep_gemm_chain_run(current_stream_ptr(), bn, split_k, iters, C.byref(ms), C.byref(levels)))
    return ms.value, levels.value


def gemm_bench(A, B, C_out, *, a_mn=False, b_mn=False, path="tc", epi=None, bn=0, split_k=0, ws=None, iters=50):
    """Average milliseconds per launch of a planned GEMM (tuning aid); returns (ms, bn, split_k)."""
    lib = load()
    M = A.shape[1] if a_mn else A.shape[0]
    K = A.shape[0] if a_mn else A.shape[1]
    N = B.shape[1] if b_mn else B.shape[0]
    epi = epi or make_epilogue()
    ms, bno, so = C.c_float(), C.c_int(), C.c_int()
    rc = lib.rlrep_gemm_bench(current_stream_ptr(), 0 if path == "tc" else 1, M, N, K, A.data_ptr(), A.stride(0),
                              int(a_mn), B.data_ptr(), B.stride(0), int(b_mn), C_out.data_ptr(), C_out.stride(0),
                              C.byref(epi), bn, split_k, ws.data_ptr() if ws is not None else None,
                              ws.numel() if ws is not None else 0, iters, C.byref(ms), C.byref(bno), C.byref(so))
    check(rc)
    return ms.value, bno.value, so.value
