"""ctypes binding of libdqgp.so (the C ABI declared in include/dqgp.h).

There is deliberately no fallback: if the library is missing or a call fails, this raises.  Build it with
``python distributed-quantum-gaussian-processes_b200/build.py`` (or ``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdqgp.so")


class DqgpError(RuntimeError):
    pass


class Gate(C.Structure):
    _fields_ = [("kind", C.c_int32), ("q0", C.c_int32), ("q1", C.c_int32), ("form", C.c_int32),
                ("pidx", C.c_int32), ("fidx", C.c_int32), ("coef", C.c_double)]


ENCODINGS = {"chebyshev": 0, "hubregtsen": 1, "yz_cx": 2, "kyriienko": 3}
# pairwisekernel = PairwiseKernel(metric="linear") = f.g, the dot product with sigma_0 = 0 (kernels.outer_hyp)
OUTER_KERNELS = {"gaussian": 0, "matern": 1, "expsinesquared": 2, "rationalquadratic": 3, "dotproduct": 4, "pairwisekernel": 4}

_vp, _i, _d, _sz = C.c_void_p, C.c_int, C.c_double, C.c_size_t
_dp = C.POINTER(C.c_double)

# name -> (restype, argtypes); every symbol include/dqgp.h declares
SIGNATURES = {
    "dqgp_version": (_i, []),
    "dqgp_last_error": (C.c_char_p, []),
    "dqgp_circuit_create": (_i, [_i, _i, _i, _i, C.POINTER(_vp)]),
    "dqgp_circuit_destroy": (None, [_vp]),
    "dqgp_circuit_num_parameters": (_i, [_vp]),
    "dqgp_circuit_num_gates": (_i, [_vp]),
    "dqgp_circuit_num_passes": (_i, [_vp]),
    "dqgp_circuit_num_passes_cx_free": (_i, [_vp]),
    "dqgp_circuit_num_fused_ops": (_i, [_vp]),
    "dqgp_circuit_shifted_u2_applications": (C.c_longlong, [_vp]),
    "dqgp_circuit_describe": (_i, [_vp, C.POINTER(Gate), _i]),
    "dqgp_features": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp]),
    "dqgp_states": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp]),
    "dqgp_features_shifted": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp]),
    "dqgp_states_shifted": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp]),
    "dqgp_gram_projected": (_i, [_i, _dp, _vp, _i, _vp, _i, _i, _vp, _i, _i, _vp]),
    "dqgp_gram_fidelity": (_i, [_vp, _i, _vp, _i, _i, _vp, _i, _i, _vp]),
    "dqgp_projected_self_kernel": (_i, [_i, _dp, _vp, _i, _i, _vp, _vp]),
    "dqgp_solver_create": (_i, [_i, C.POINTER(_vp)]),
    "dqgp_solver_create_ex": (_i, [_i, _i, C.POINTER(_vp)]),
    "dqgp_solver_create_lean": (_i, [_i, _i, C.POINTER(_vp)]),
    "dqgp_solver_is_lean": (_i, [_vp]),
    "dqgp_solver_destroy": (None, [_vp]),
    "dqgp_solver_n": (_i, [_vp]),
    "dqgp_solver_ld": (_i, [_vp]),
    "dqgp_solver_matrix": (_vp, [_vp]),
    "dqgp_solver_inverse": (_vp, [_vp]),
    "dqgp_solver_factor": (_vp, [_vp]),
    "dqgp_solver_bytes": (_sz, [_vp]),
    "dqgp_solver_potrf_launches": (_i, [_vp]),
    "dqgp_add_diagonal": (_i, [_vp, _i, _i, _d, _vp]),
    "dqgp_potrf_solve_inv": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "dqgp_solver_quadform_rows": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "dqgp_solver_quadform_rows_inplace": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "dqgp_solver_apply_factor": (_i, [_vp, _vp, _vp, _vp]),
    "dqgp_lu_workspace_bytes": (_sz, [_i]),
    "dqgp_lu_solve_inv": (_i, [_vp, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "dqgp_dgemm_general": (_i, [_i, _i, _i, _d, _vp, _i, _vp, _i, _d, _vp, _i, _vp]),
    "dqgp_rowdot": (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _vp]),
    "dqgp_dgemm": (_i, [_i, _i, _i, _i, _i, _d, _vp, _i, _vp, _i, _d, _vp, _i, _vp]),
    "dqgp_shift_parameter_sets": (_i, [_vp, _i, _d, _d, _vp, _vp]),
    "dqgp_grad_workspace_bytes": (_sz, [_i, _i]),
    "dqgp_grad_projected": (_i, [_i, _dp, _vp, _i, _vp, _vp, _i, _i, _i, _d, _vp, _vp, _vp]),
    "dqgp_grad_fidelity": (_i, [_vp, _i, _vp, _vp, _i, _i, _i, _d, _vp, _vp, _vp]),
    "dqgp_features_jacobian": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "dqgp_states_jacobian": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "dqgp_grad_fidelity_analytic_workspace_bytes": (_sz, [_i, _i]),
    "dqgp_grad_fidelity_analytic": (_i, [_vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "dqgp_grad_analytic_workspace_bytes": (_sz, [_i, _i]),
    "dqgp_grad_projected_analytic": (_i, [_i, _dp, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "dqgp_grad_outer_hyperparameters_workspace_bytes": (_sz, [_i]),
    "dqgp_grad_outer_hyperparameters": (_i, [_i, _dp, _vp, _i, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "dqgp_grad_noise_std": (_i, [_vp, _i, _vp, _i, _d, _vp, _vp]),
    "dqgp_nll_terms": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "dqgp_admm_local": (_i, [_vp, _vp, _vp, _i, _d, _d, _d, _vp, _vp, _vp]),
    "dqgp_admm_consensus": (_i, [_vp, _vp, _i, _i, _d, _d, _vp, _vp]),
    "dqgp_admm_consensus_strided": (_i, [_vp, _vp, _i, _i, _i, _d, _d, _vp, _vp]),
    "dqgp_predict_mean": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp]),
    "dqgp_predict_finish": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
}

_lib = None


def load():
    """Load libdqgp.so and declare every signature.  Raises DqgpError when the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        # not a fallback: the same CUDA sources are compiled on the spot when the toolkit is present
        try:
            import importlib.util
            spec = importlib.util.spec_from_file_location("_dqgp_build", os.path.join(HERE, "build.py"))
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            mod.build()
        except Exception as exc:
            raise DqgpError(f"{LIB_PATH} not found and building it failed ({exc}); build it with "
                            f"`python {os.path.join(HERE, 'build.py')}` (nvcc, sm_100a). dqgp_b200 has no CPU fallback.") from exc
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError here = header / library drift
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc is not None and rc < 0:
        msg = load().dqgp_last_error()
        raise DqgpError(f"{what}: {msg.decode() if msg else 'error ' + str(rc)}")
    return rc


def hyp_array(values):
    return (C.c_double * len(values))(*values)
