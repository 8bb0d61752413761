"""GP prediction, NLPD and k-fold CV on the consensus parameters with the reference's signatures
(``main.predict_quantum_gp`` main.py:1364-1488, NLPD main.py:1546-1552, ``k_fold_cross_validation_consensus``
main.py:1490-1596).  K(train,train) goes straight into the solver, K(test,train) is a rectangular Gram,
the predictive variance uses v = L^-1 K(test,train)^T through the DMMA GEMM, and — unlike the reference,
which evaluates the full K(test,test) and keeps its diagonal (main.py:1430,1463) — only the diagonal
k(x*,x*) is evaluated.  KFold orchestration stays on the host (scikit-learn), as in the reference.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from ._lib import check
from .engine import Solver
from .kernels import create_quantum_kernel, dev_f64, stream_ptr


def predict_quantum_gp(X_train, Y_train, X_test, quantum_kernel_params, num_qubits, num_layers, noise_std,
                       use_parameter_shift=True, encoding_type="yz_cx", kernel_type="fidelity", measurement="XYZ",
                       outer_kernel="gaussian", outer_kernel_params=None, regularization=None, return_kernels=False,
                       Y_test=None, lean=None):
    """-> (mean, var, K_tt, K_st, K_ss); the three matrices are None unless ``return_kernels`` (they are only
    used for plots in the reference).  With ``Y_test`` the mean NLPD is computed on the device and attached as
    ``predict_quantum_gp.last_nlpd``.

    ``lean`` (None = decide from free HBM): factor K(train,train) in place with ONE padded square, alpha by blocked
    substitution and the predictive variance by in-place forward substitution on K(test,train) - the path for
    training sets whose three-square workspace does not fit (config 5: 117964 samples = 112 GB per square)."""
    lib = _lib.load()
    X_train = np.asarray(X_train, dtype=np.float64)
    X_test = np.asarray(X_test, dtype=np.float64)
    if X_train.ndim == 1:
        X_train = X_train.reshape(-1, 1)
    if X_test.ndim == 1:
        X_test = X_test.reshape(-1, 1)
    d = X_train.shape[1]
    qk = create_quantum_kernel(num_qubits, d, num_layers, use_parameter_shift, encoding_type, kernel_type, measurement,
                               outer_kernel, outer_kernel_params, regularization)
    qk.assign_parameters(quantum_kernel_params)
    n, nt = X_train.shape[0], X_test.shape[0]
    d_xtr, d_xte = dev_f64(X_train), dev_f64(X_test)
    d_p = dev_f64(np.asarray(quantum_kernel_params, dtype=np.float64).reshape(1, -1))
    d_y = dev_f64(np.asarray(Y_train, dtype=np.float64).reshape(-1))
    st = stream_ptr()
    if lean is None:
        npad = -(-n // 128) * 128
        free, _ = torch.cuda.mem_get_info()
        lean = 3 * 8 * npad * npad + 8 * nt * n > 0.9 * free
    if lean and return_kernels:
        raise ValueError("return_kernels is not available on the lean path (K(test,train) is overwritten in place)")
    solver = Solver(n, lean=bool(lean))
    k_tt = solver.matrix()
    # same=2: only the lower tiles are written (all the factorisation reads) unless the caller wants K back
    qk.evaluate_device(d_xtr, d_xtr, d_p, same=True if return_kernels else 2, out=k_tt, ld=solver.ld)
    k_tt_host = k_tt.cpu().numpy() if return_kernels else None
    # K + sigma^2 I, then + 1e-6 I as two separate additions (main.py:1434-1438)
    check(lib.dqgp_add_diagonal(solver.matrix_ptr, n, solver.ld, float(noise_std) ** 2, st), "add diagonal")
    check(lib.dqgp_add_diagonal(solver.matrix_ptr, n, solver.ld, 1e-6, st), "add diagonal")
    f64 = dict(dtype=torch.float64, device=d_xtr.device)
    alpha, logdet = torch.empty(n, **f64), torch.zeros(1, **f64)
    info = torch.zeros(1, dtype=torch.int32, device=d_xtr.device)
    check(lib.dqgp_potrf_solve_inv(solver.handle, d_y.data_ptr(), alpha.data_ptr(), logdet.data_ptr(), info.data_ptr(), 0, st),
          "potrf")
    mean, var = torch.empty(nt, **f64), torch.empty(nt, **f64)
    if lean:
        # K(test,train) in a padded buffer (rows to a multiple of 128, leading dimension = the solver's), mean first,
        # then the rows are overwritten by (L^-1 k_i)^T
        ntp, ldk = -(-nt // 128) * 128, solver.ld
        k_st = torch.empty((ntp, ldk), **f64)
        k_st[nt:].zero_()
        k_st[:, n:].zero_()
        qk.evaluate_device(d_xte, d_xtr, d_p, same=False, out=k_st, ld=ldk)
        check(lib.dqgp_predict_mean(k_st.data_ptr(), nt, n, ldk, alpha.data_ptr(), mean.data_ptr(), st), "predict mean")
        quad = torch.empty(ntp, **f64)
        check(lib.dqgp_solver_quadform_rows_inplace(solver.handle, k_st.data_ptr(), ntp, ldk, quad.data_ptr(), st), "quadform")
        kst_ptr, ldk_arg = None, 0
    else:
        k_st = qk.evaluate_device(d_xte, d_xtr, d_p, same=False)
        quad = torch.empty(nt, **f64)
        check(lib.dqgp_solver_quadform_rows(solver.handle, k_st.data_ptr(), nt, n, quad.data_ptr(), st), "quadform")
        kst_ptr, ldk_arg = k_st.data_ptr(), n
    # diag K(test,test): each test point against itself (1 x 1 Grams batched as a diagonal extraction)
    kss_diag = _self_kernel_diag(qk, d_xte, d_p)
    nlpd_buf = torch.empty(1 + nt, **f64) if Y_test is not None else None
    d_yt = dev_f64(np.asarray(Y_test, dtype=np.float64).reshape(-1)) if Y_test is not None else None
    check(lib.dqgp_predict_finish(kst_ptr, nt, n, ldk_arg, alpha.data_ptr(), kss_diag.data_ptr(), quad.data_ptr(),
                                  d_yt.data_ptr() if d_yt is not None else None, mean.data_ptr(), var.data_ptr(),
                                  nlpd_buf.data_ptr() if nlpd_buf is not None else None, st), "predict finish")
    if int(info.item()) != 0:
        # np.linalg.cholesky raised in the reference: its except-branch inverts directly (main.py:1479-1486):
        #   a_inv = np.linalg.inv(K);  alpha = a_inv @ y;  mean = K_st @ alpha;  var = max(diag(K_ss - K_st a_inv K_st^T), 1e-10)
        # np.linalg.inv is a partial-pivoting LU (getrf + getri): the same factorisation runs here on the device.
        if lean:
            raise RuntimeError("Cholesky failed: training kernel matrix is not positive definite, and the LU fallback "
                               "(main.py:1479-1486) needs the three-square workspace: call with lean=False")
        qk.evaluate_device(d_xtr, d_xtr, d_p, same=True, out=k_tt, ld=solver.ld)           # both triangles
        check(lib.dqgp_add_diagonal(solver.matrix_ptr, n, solver.ld, float(noise_std) ** 2, st), "add diagonal")
        check(lib.dqgp_add_diagonal(solver.matrix_ptr, n, solver.ld, 1e-6, st), "add diagonal")
        work = torch.empty(int(lib.dqgp_lu_workspace_bytes(n)) // 8 + 2, **f64)
        check(lib.dqgp_lu_solve_inv(solver.matrix_ptr, solver.ld, n, None, None, solver.inverse_ptr, solver.ld, None, work.data_ptr(), st),
              "lu fallback")
        check(lib.dqgp_dgemm_general(n, 1, n, 1.0, solver.inverse_ptr, solver.ld, d_y.data_ptr(), 1, 0.0, alpha.data_ptr(), 1, st),
              "alpha = A^-1 y")
        t_rows = torch.empty((nt, n), **f64)
        check(lib.dqgp_dgemm_general(nt, n, n, 1.0, k_st.data_ptr(), n, solver.inverse_ptr, solver.ld, 0.0, t_rows.data_ptr(), n, st),
              "K_st A^-1")
        check(lib.dqgp_rowdot(t_rows.data_ptr(), n, k_st.data_ptr(), n, nt, n, quad.data_ptr(), st), "diag(K_st A^-1 K_st^T)")
        check(lib.dqgp_predict_finish(kst_ptr, nt, n, ldk_arg, alpha.data_ptr(), kss_diag.data_ptr(), quad.data_ptr(),
                                      d_yt.data_ptr() if d_yt is not None else None, mean.data_ptr(), var.data_ptr(),
                                      nlpd_buf.data_ptr() if nlpd_buf is not None else None, st), "predict finish")
        predict_quantum_gp.used_lu_fallback = True
    predict_quantum_gp.last_nlpd = float(nlpd_buf[0].item()) if nlpd_buf is not None else None
    k_ss = qk.evaluate_device(d_xte, d_xte, d_p, same=True).cpu().numpy() if return_kernels else None
    return (mean.cpu().numpy(), var.cpu().numpy(), k_tt_host, k_st.cpu().numpy() if return_kernels else None, k_ss)


predict_quantum_gp.last_nlpd = None
predict_quantum_gp.used_lu_fallback = False


def _self_kernel_diag(qk, d_x, d_p):
    """k(x_i, x_i) for every row: outer(f_i, f_i) for the projected kernels (exactly 1 for the stationary ones, sigma_0^2 + |f_i|^2
    for the dot product); |<psi|psi>|^2 for fidelity."""
    nt = d_x.shape[0]
    if hasattr(qk, "outer_kernel"):
        out = torch.empty(nt, dtype=torch.float64, device=d_x.device)
        outer_id, m = _lib.OUTER_KERNELS[qk.outer_kernel], 3 * qk.encoding_circuit.num_qubits
        # only the dot product reads the features (the stationary kernels' k(f, f) is 1 whatever f is)
        f = qk.encoding_circuit.features(d_x, d_p) if outer_id == _lib.OUTER_KERNELS["dotproduct"] else None     # (1, nt, 3q)
        check(_lib.load().dqgp_projected_self_kernel(outer_id, _lib.hyp_array(qk._hyp), f.data_ptr() if f is not None else None, nt, m,
                                                     out.data_ptr(), stream_ptr()), "dqgp_projected_self_kernel")
        return out
    s = qk.encoding_circuit.states(d_x, d_p)[0]           # (nt, dim, 2)
    nrm = (s * s).sum(dim=(1, 2))
    return nrm * nrm


def gather_fold_scores(scores, process_group, rank, world_size):
    """All-gather the (k_folds, 3) score table: row f is taken from its owner, rank f % world_size."""
    import torch.distributed as dist
    backend = dist.get_backend(process_group)
    dev = torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu")
    mine = torch.from_numpy(np.ascontiguousarray(scores)).to(dev)
    allr = torch.empty((world_size,) + tuple(mine.shape), dtype=mine.dtype, device=dev)
    dist.all_gather_into_tensor(allr.view(-1), mine.view(-1), group=process_group)
    allr = allr.cpu().numpy()
    return np.stack([allr[f % world_size, f] for f in range(scores.shape[0])])


def nlpd(Y_true, y_pred_mean, y_pred_var):
    """Mean negative log predictive density, main.py:1546-1552 (host formula for host arrays)."""
    var = np.maximum(np.asarray(y_pred_var, dtype=np.float64), 1e-10)
    r = np.asarray(Y_true, dtype=np.float64) - np.asarray(y_pred_mean, dtype=np.float64)
    return float(np.mean(0.5 * np.log(2 * np.pi) + 0.5 * np.log(var) + 0.5 * (r ** 2 / var)))


def k_fold_cross_validation_consensus(X_train, Y_train, consensus_params, num_qubits, num_layers, noise_std, k_folds=5,
                                      use_parameter_shift=True, encoding_type="yz_cx", kernel_type="fidelity",
                                      measurement="XYZ", outer_kernel="gaussian", outer_kernel_params=None,
                                      regularization=None, random_seed=42, process_group=None, rank=0, world_size=1,
                                      _predict=None):
    """Same result dict as main.py:1490-1596 (mean/std NLPD, R^2, RMSE over valid folds).

    With ``world_size`` > 1 (one process per GPU) the folds - independent factorisations - are dealt round-robin to the
    ranks (fold f on rank f % world_size) and the three per-fold scores are all-gathered, so every rank returns the
    same dict as a single process would; no training data crosses NVLink."""
    from sklearn.metrics import mean_squared_error, r2_score
    from sklearn.model_selection import KFold

    X_train = np.asarray(X_train, dtype=np.float64)
    Y_train = np.asarray(Y_train, dtype=np.float64)
    predict = _predict or predict_quantum_gp
    scores = np.full((k_folds, 3), np.nan)
    for f, (tr, va) in enumerate(KFold(n_splits=k_folds, shuffle=True, random_state=random_seed).split(X_train)):
        if f % world_size != rank:
            continue
        try:
            mean, var, _, _, _ = predict(X_train[tr], Y_train[tr], X_train[va], consensus_params, num_qubits,
                                         num_layers, noise_std, use_parameter_shift, encoding_type, kernel_type,
                                         measurement, outer_kernel, outer_kernel_params, regularization)
            scores[f] = (nlpd(Y_train[va], mean, var), r2_score(Y_train[va], mean),
                         float(np.sqrt(mean_squared_error(Y_train[va], mean))))
        except Exception:
            scores[f] = (float("inf"), -float("inf"), float("inf"))
    if world_size > 1:
        scores = gather_fold_scores(scores, process_group, rank, world_size)
    fold_nlpds, fold_r2s, fold_rmses = [list(map(float, scores[:, c])) for c in range(3)]
    valid = [v for v in fold_nlpds if not np.isinf(v)]
    if len(valid) >= k_folds // 2:
        ok = [not np.isinf(v) for v in fold_nlpds]
        out = {"mean_nlpd": float(np.mean(valid)), "std_nlpd": float(np.std(valid)),
               "mean_r2": float(np.mean([r for r, o in zip(fold_r2s, ok) if o])),
               "mean_rmse": float(np.mean([r for r, o in zip(fold_rmses, ok) if o]))}
    else:
        out = {"mean_nlpd": float("inf"), "std_nlpd": float("inf"), "mean_r2": -float("inf"), "mean_rmse": float("inf")}
    out.update({"fold_nlpds": fold_nlpds, "fold_r2s": fold_r2s, "fold_rmses": fold_rmses, "valid_folds": len(valid),
                "total_folds": k_folds})
    return out
