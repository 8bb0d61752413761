"""GPU parity of the RationalQuadratic, DotProduct and PairwiseKernel outer kernels of the projected kernel (the rest of the
reference's --outer-kernel choices, main.py:1996-2013) against scikit-learn and the oracle: the Gram kernels, k(f, f), the
fused central-difference gradient, the agent step that honours the outer kernel, prediction / k-fold CV, the ADMM driver at
the Q1 default, and the quantum-GP dataset sampler.  The oracle's agent step, prediction and driver evaluate the new outer
kernels with the scikit-learn classes (``sklearn_oracle`` installs test_oracle_outer_kernels.sklearn_outer_kernel_matrix)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
sk = pytest.importorskip("sklearn.gaussian_process.kernels")

NEW = ["rationalquadratic", "dotproduct", "pairwisekernel"]
SKLEARN = {"rationalquadratic": lambda: sk.RationalQuadratic(), "dotproduct": lambda: sk.DotProduct(),
           "pairwisekernel": lambda: sk.PairwiseKernel(metric="linear"),
           "gaussian": lambda: sk.RBF(length_scale=1.0 / np.sqrt(2.0)), "matern": lambda: sk.Matern(nu=1.5),
           "expsinesquared": lambda: sk.ExpSineSquared()}


@pytest.fixture(scope="module")
def d():
    import dqgp_b200
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")
    return dqgp_b200


@pytest.fixture
def sklearn_oracle(monkeypatch):
    from oracle import qkernels
    from test_oracle_outer_kernels import sklearn_outer_kernel_matrix
    monkeypatch.setattr(qkernels, "outer_kernel_matrix", sklearn_outer_kernel_matrix)


def _sp():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _gram(d, outer, hyp, F, G, same, ld_extra=3, sentinel=-7.0):
    """dqgp_gram_projected into an (n1, n2 + ld_extra) buffer filled with `sentinel`; same != 0 passes F for both operands."""
    from dqgp_b200 import _lib
    n1, n2, m = F.shape[0], G.shape[0], F.shape[1]
    K = torch.full((n1, n2 + ld_extra), sentinel, dtype=torch.float64, device="cuda")
    dF = d.kernels.dev_f64(F)
    dG = dF if same else d.kernels.dev_f64(G)
    lib = d.load()
    rc = lib.dqgp_gram_projected(_lib.OUTER_KERNELS[outer], _lib.hyp_array(hyp), dF.data_ptr(), n1, dG.data_ptr(), n2, m,
                                 K.data_ptr(), n2 + ld_extra, same, _sp())
    assert rc == 0, lib.dqgp_last_error()
    torch.cuda.synchronize()
    return K.cpu().numpy()


def _check_entries(outer, K, ref, F, G, sigma0_sq=None, mask=None):
    """RationalQuadratic to 1e-10 relative; dot products to 1e-13 (sigma_0^2 + |f||g|): entries near 0 make a relative bar
    meaningless there, the bound is the size of the summands.  `mask` selects the entries compared (default: all)."""
    mask = np.ones(K.shape, dtype=bool) if mask is None else mask
    if outer == "rationalquadratic":
        assert np.max(np.abs(K - ref)[mask] / np.abs(ref)[mask]) <= 1e-10
    else:
        s2 = (1.0 if outer == "dotproduct" else 0.0) if sigma0_sq is None else sigma0_sq
        scale = s2 + np.outer(np.linalg.norm(F, axis=1), np.linalg.norm(G, axis=1))
        assert np.all((np.abs(K - ref) <= 1e-13 * scale)[mask])


@pytest.mark.parametrize("outer", NEW)
@pytest.mark.parametrize("m", [9, 24])
def test_gram_matches_sklearn_ragged_shapes(d, outer, m):
    """Rectangular tiles at ragged sizes with ld > n2 (nothing written past the logical width), and the two symmetric modes:
    same = 1 (lower tiles + mirror) and same = 2 (lower tiles only).  RationalQuadratic gives exactly 1 on duplicate samples
    and on the diagonal; the dot products' diagonal is sigma_0^2 + |f|^2."""
    rng = np.random.default_rng(m)
    k = SKLEARN[outer]()
    hyp = d.kernels.outer_hyp(outer)
    for n1, n2 in [(1, 1), (63, 65), (65, 63), (129, 1), (1, 129), (129, 65)]:
        F, G = rng.uniform(-1, 1, (n1, m)), rng.uniform(-1, 1, (n2, m))
        nd = min(3, n1, n2)
        G[-nd:] = F[:nd]                                         # exact duplicates: F[i] == G[n2 - nd + i]
        K = _gram(d, outer, hyp, F, G, 0)
        ref = k(F, G)
        _check_entries(outer, K[:, :n2], ref, F, G)
        assert np.all(K[:, n2:] == -7.0)
        if outer == "rationalquadratic":
            assert np.all(K[:nd, n2 - nd:].diagonal() == 1.0)
    for n in [1, 63, 65, 129]:
        F = rng.uniform(-1, 1, (n, m))
        if n > 2:
            F[2] = F[0]                                          # a duplicate inside the symmetric Gram
        ref = k(F)                                               # scikit-learn's symmetric call, Y = None
        for same in (1, 2):
            K = _gram(d, outer, hyp, F, F, same)
            assert np.all(K[:, n:] == -7.0)
            # same = 2 leaves the 64 x 64 tiles above the diagonal unwritten: compare the lower triangle
            _check_entries(outer, K[:, :n], ref, F, F, mask=None if same == 1 else np.tril(np.ones((n, n), dtype=bool)))
            if same == 1:
                assert np.array_equal(K[:, :n], K[:, :n].T)      # the mirror is exact
            if outer == "rationalquadratic":
                assert np.all(np.diagonal(K[:, :n]) == 1.0)
                if n > 2:
                    assert K[2, 0] == 1.0
            else:
                nrm2 = np.einsum("ij,ij->i", F, F) + (1.0 if outer == "dotproduct" else 0.0)
                assert np.allclose(np.diagonal(K[:, :n]), nrm2, rtol=1e-14, atol=0)


def test_gram_rational_quadratic_general_alpha_and_dot_product_sigma(d):
    """alpha != 1 takes the exp(-alpha log(base)) branch; sigma_0 != 1 through the ABI; validation of the new hyper-parameters."""
    from dqgp_b200 import _lib
    rng = np.random.default_rng(11)
    F, G = rng.uniform(-1, 1, (130, 15)), rng.uniform(-1, 1, (67, 15))
    K = _gram(d, "rationalquadratic", [0.7, 2.5], F, G, 0)[:, :67]
    ref = sk.RationalQuadratic(length_scale=0.7, alpha=2.5)(F, G)
    assert np.max(np.abs(K - ref) / np.abs(ref)) <= 1e-10
    Ks = _gram(d, "rationalquadratic", [0.7, 2.5], F, F, 1)[:, :130]
    assert np.max(np.abs(Ks - sk.RationalQuadratic(length_scale=0.7, alpha=2.5)(F)) / Ks) <= 1e-10
    assert np.all(np.diagonal(Ks) == 1.0)
    K = _gram(d, "dotproduct", [0.3], F, G, 0)[:, :67]
    _check_entries("dotproduct", K, sk.DotProduct(sigma_0=0.3)(F, G), F, G, sigma0_sq=0.09)
    lib = d.load()
    buf = torch.zeros((4, 4), dtype=torch.float64, device="cuda")
    f = d.kernels.dev_f64(F[:4])
    for outer, hyp, msg in [(3, [0.0, 1.0], b"length_scale and alpha"), (3, [1.0, -1.0], b"length_scale and alpha"),
                            (4, [-0.5], b"sigma_0"), (5, [1.0], b"unknown outer kernel")]:
        assert lib.dqgp_gram_projected(outer, _lib.hyp_array(hyp), f.data_ptr(), 4, f.data_ptr(), 4, 15, buf.data_ptr(), 4, 0, _sp()) < 0
        assert msg in lib.dqgp_last_error()


@pytest.mark.parametrize("outer", NEW)
def test_gram_nan_features_propagate(d, outer):
    """A NaN feature (arccos outside [-1, 1]) makes its sample's row and column NaN, as in NumPy, and nothing else."""
    rng = np.random.default_rng(3)
    F = rng.uniform(-1, 1, (70, 9))
    F[5, 4] = np.nan
    G = rng.uniform(-1, 1, (66, 9))
    hyp = d.kernels.outer_hyp(outer)
    K = _gram(d, outer, hyp, F, G, 0)[:, :66]
    assert np.all(np.isnan(K[5]))
    assert np.all(np.isfinite(np.delete(K, 5, axis=0)))
    for same in (1, 2):
        K = _gram(d, outer, hyp, F, F, same)[:, :70]
        low = np.tril(np.ones((70, 70), dtype=bool))
        bad = np.zeros((70, 70), dtype=bool)
        bad[5, :] = bad[:, 5] = True
        assert np.all(np.isnan(K[bad & low]))
        assert np.all(np.isfinite(K[~bad & low]))


@pytest.mark.parametrize("outer", ["gaussian", "matern", "expsinesquared"] + NEW)
def test_projected_self_kernel_equals_sklearn_diag(d, outer):
    from dqgp_b200 import _lib
    rng = np.random.default_rng(4)
    lib = d.load()
    for n, m in [(1, 3), (257, 24), (1000, 30)]:
        F = rng.uniform(-1, 1, (n, m))
        out = torch.full((n,), -1.0, dtype=torch.float64, device="cuda")
        rc = lib.dqgp_projected_self_kernel(_lib.OUTER_KERNELS[outer], _lib.hyp_array(d.kernels.outer_hyp(outer)),
                                            d.kernels.dev_f64(F).data_ptr(), n, m, out.data_ptr(), _sp())
        assert rc == 0, lib.dqgp_last_error()
        torch.cuda.synchronize()
        got, ref = out.cpu().numpy(), SKLEARN[outer]().diag(F)
        if outer in ("dotproduct", "pairwisekernel"):
            assert np.allclose(got, ref, rtol=1e-14, atol=0)
        else:
            assert np.array_equal(got, ref) and np.all(got == 1.0)
    out = torch.empty(4, dtype=torch.float64, device="cuda")
    assert lib.dqgp_projected_self_kernel(3, None, None, 4, 9, out.data_ptr(), _sp()) == 0        # stationary: F not read
    assert lib.dqgp_projected_self_kernel(4, None, None, 4, 9, out.data_ptr(), _sp()) < 0
    assert lib.dqgp_projected_self_kernel(4, _lib.hyp_array([0.5]), d.kernels.dev_f64(np.full((4, 9), 0.5)).data_ptr(), 4, 9,
                                          out.data_ptr(), _sp()) == 0
    torch.cuda.synchronize()
    assert np.allclose(out.cpu().numpy(), 0.25 + 9 * 0.25, rtol=1e-15, atol=0)


def _engine(d, enc, q, dd, layers, n, outer, seed):
    x, y = d.synthetic_dataset(n, dd, enc, seed=seed)
    eng = d.AgentEngine(x, y, encoding_type=enc, kernel_type="projected", num_qubits=q, num_layers=layers, noise_std=0.1, rho=100.0,
                        L=100.0, outer_kernel=outer, training_ignores_outer_kernel=False)
    return x, y, eng


@pytest.mark.parametrize("outer", ["rationalquadratic", "dotproduct"])
@pytest.mark.parametrize("enc,q,dd,layers,n", [("kyriienko", 4, 6, 2, 150), ("chebyshev", 3, 2, 1, 97), ("yz_cx", 5, 4, 2, 200),
                                                ("hubregtsen", 3, 4, 2, 64)])
def test_fused_gradient_new_outer_kernels_match_oracle(d, sklearn_oracle, outer, enc, q, dd, layers, n):
    """dqgp_grad_projected on the ORACLE's C^-1 and alpha equals 1/2 sum(B o dK_i^T) with the oracle's materialised dK
    (agent_riemannian.py:431-436) to 1e-8, and so does the whole device path (Cholesky, alpha, inverse, NLL).  The dot
    product's diagonal carries gradient.  Even m (kyriienko, q = 4) stages through the tensor map; the same features at an
    8-byte offset take the cp.async kernel, which must give the same gradient to the last bit."""
    from oracle import agent_step
    x, y, eng = _engine(d, enc, q, dd, layers, n, outer, n)
    cfg = agent_step.KernelConfig(enc, "projected", q, layers, outer, training_ignores_outer_kernel=False)
    z = np.round(np.random.RandomState(n).rand(eng.P) * np.pi, 4)
    K, dK = agent_step.kernel_and_derivatives(cfg, x, np.mod(z, np.pi), np.pi / 8)
    if outer == "dotproduct":
        assert np.max(np.abs(np.diagonal(dK, axis1=1, axis2=2))) > 1e-3           # the diagonal is not constant
    grad_ref, comp, _, alpha, cinv = agent_step.gp_terms(K, dK, y, 0.1, want_cond=False)
    eng.simulate(d.kernels.dev_f64(z))
    eng.gram()
    Kd = torch.tril(eng.solver.matrix()).cpu().numpy()
    ref_l = np.tril(K + 0.01 * np.eye(n))
    if outer == "rationalquadratic":
        assert np.max(np.abs(Kd - ref_l) / np.maximum(np.abs(ref_l), 1e-300)) < 1e-10
    else:
        assert np.max(np.abs(Kd - ref_l)) < 1e-13 * np.abs(ref_l).max()
    eng.solver.inverse().copy_(torch.from_numpy(cinv).cuda())
    eng.d_alpha.copy_(torch.from_numpy(alpha).cuda())
    eng.gradient()
    torch.cuda.synchronize()
    got = eng.d_grad.cpu().numpy().copy()
    tol = 1e-8 * max(1.0, np.abs(grad_ref).max())
    assert np.max(np.abs(got - grad_ref)) < tol
    # the cp.async staging path on the same operands
    lib, s = d.load(), eng.solver
    buf = torch.empty(eng.d_feat.numel() + 1, dtype=torch.float64, device="cuda")
    feat = buf[1:].view(eng.d_feat.shape)
    feat.copy_(eng.d_feat)
    assert feat.data_ptr() % 16 == 8
    grad = torch.zeros_like(eng.d_grad)
    assert lib.dqgp_grad_projected(eng._outer_id, eng._hyp, s.inverse_ptr, s.ld, eng.d_alpha.data_ptr(), feat.data_ptr(), n, eng.m,
                                   eng.P, eng.h, grad.data_ptr(), eng.d_work.data_ptr(), _sp()) == 0, lib.dqgp_last_error()
    torch.cuda.synchronize()
    assert np.array_equal(got, grad.cpu().numpy())
    # the whole device path
    eng.factor(); eng.gradient()
    torch.cuda.synchronize(); eng.check_info()
    assert np.max(np.abs(eng.d_grad.cpu().numpy() - grad_ref)) < tol
    assert abs(float(eng.d_nll[3].item()) - comp["total"]) < 1e-8 * max(1.0, abs(comp["total"]))


@pytest.mark.parametrize("outer", NEW)
def test_agent_step_honouring_the_outer_kernel_matches_oracle(d, sklearn_oracle, outer):
    """RiemannianAgent.train_and_update with training_ignores_outer_kernel=False against agent_step.train_and_update: theta and
    psi on the same 1e-4 grid point, NLL to 1e-8."""
    from oracle import agent_step
    enc, q, layers, dd, n = "chebyshev", 4, 2, 2, 180
    x, y = d.synthetic_dataset(n, dd, enc, seed=5)
    cfg = agent_step.KernelConfig(enc, "projected", q, layers, outer, training_ignores_outer_kernel=False)
    ag = d.RiemannianAgent("a", x, y, q, 0.1, 100.0, 100.0, use_parameter_shift=True, num_layers=layers, encoding_type=enc,
                           kernel_type="projected", outer_kernel=outer, training_ignores_outer_kernel=False)
    from oracle import circuits
    rs = np.random.RandomState(8)
    P = circuits.num_parameters(enc, q, layers)
    z, psi = np.round(rs.rand(P), 4), np.round(rs.rand(P), 4)
    theta, psi_new, nll, _, _ = ag.train_and_update(z, psi)
    ref = agent_step.train_and_update(cfg, x, y, z, psi, 0.1, 100.0, 100.0, want_cond=False)
    assert np.max(np.abs(ag.last_gradient - ref.grad)) < 1e-8 * max(1.0, np.abs(ref.grad).max())
    assert np.max(np.abs(theta - ref.theta)) < 1e-12 and np.max(np.abs(psi_new - ref.psi)) < 1e-9
    assert abs(nll - ref.nll) < 1e-8 * max(1.0, abs(ref.nll))


@pytest.mark.parametrize("outer", NEW)
def test_predict_and_cv_match_oracle(d, sklearn_oracle, outer):
    """predict_quantum_gp (three-square and lean) and k_fold_cross_validation_consensus against oracle.driver.predict / nlpd with
    the same KFold splits: mean and variance to 1e-8, NLPD to 1e-7.  The dot products' k(x*, x*) is sigma_0^2 + |f|^2."""
    from sklearn.model_selection import KFold
    from oracle import agent_step, circuits, driver
    enc, q, layers, dd = "yz_cx", 3, 2, 2
    x, y = d.synthetic_dataset(260, dd, enc, seed=9)
    xtr, ytr, xte, yte = x[:200], y[:200], x[200:], y[200:]
    P = circuits.num_parameters(enc, q, layers)
    params = np.round(np.random.RandomState(2).rand(P) * np.pi, 4)
    cfg = agent_step.KernelConfig(enc, "projected", q, layers, outer)
    ref_mean, ref_var = driver.predict(cfg, xtr, ytr, xte, params, 0.1)
    ref_nlpd = driver.nlpd(yte, ref_mean, ref_var)
    for lean in (False, True):
        mean, var, *_ = d.predict_quantum_gp(xtr, ytr, xte, params, q, layers, 0.1, True, enc, "projected", "XYZ", outer,
                                             Y_test=yte, lean=lean)
        assert np.max(np.abs(mean - ref_mean)) < 1e-8 * max(1.0, np.abs(ref_mean).max())
        assert np.max(np.abs(var - ref_var)) < 1e-8
        assert abs(d.predict_quantum_gp.last_nlpd - ref_nlpd) < 1e-7
    out = d.k_fold_cross_validation_consensus(x, y, params, q, layers, 0.1, k_folds=5, encoding_type=enc, kernel_type="projected",
                                              outer_kernel=outer, random_seed=17)
    ref_folds = []
    for tr, va in KFold(n_splits=5, shuffle=True, random_state=17).split(x):
        m_, v_ = driver.predict(cfg, x[tr], y[tr], x[va], params, 0.1)
        ref_folds.append(driver.nlpd(y[va], m_, v_))
    assert out["valid_folds"] == 5
    assert np.max(np.abs(np.array(out["fold_nlpds"]) - np.array(ref_folds))) < 1e-7
    assert abs(out["mean_nlpd"] - float(np.mean(ref_folds))) < 1e-7


def test_run_admm_rational_quadratic_at_the_q1_default(d, sklearn_oracle):
    """Under Q1 the training Grams ignore --outer-kernel: run_admm with "rationalquadratic" walks exactly the z / theta / psi
    of the "gaussian" run, and only the per-iteration CV (which honours the outer kernel) differs - it equals the oracle's."""
    from sklearn.model_selection import KFold
    from oracle import agent_step, circuits, driver
    enc, q, layers, dd = "chebyshev", 3, 1, 2
    x, y = d.synthetic_dataset(300, dd, enc, seed=21)
    shards = [(x[:100], y[:100]), (x[100:200], y[100:200])]
    cv_x, cv_y = x[200:], y[200:]
    P = circuits.num_parameters(enc, q, layers)
    rs = np.random.RandomState(4)
    theta0, psi0 = np.round(rs.rand(2, P), 4), np.round(rs.rand(2, P), 4)
    kw = dict(encoding_type=enc, kernel_type="projected", num_qubits=q, num_layers=layers, noise_std=0.1, rho=100.0, L=100.0,
              max_iter=3, theta0=theta0, psi0=psi0, cv_data=(cv_x, cv_y), cv_folds=5, seed=42)
    rq = d.run_admm(shards, outer_kernel="rationalquadratic", **kw)
    ga = d.run_admm(shards, outer_kernel="gaussian", **kw)
    assert rq["iterations"] == ga["iterations"] == 3
    for hr, hg in zip(rq["history"], ga["history"]):
        for key in ("z", "theta", "psi", "nll"):
            assert np.array_equal(hr[key], hg[key]), key
    cfg = agent_step.KernelConfig(enc, "projected", q, layers, "rationalquadratic")
    for it, h in enumerate(rq["history"], start=1):
        ref = []
        for tr, va in KFold(n_splits=5, shuffle=True, random_state=42 + it).split(cv_x):
            m_, v_ = driver.predict(cfg, cv_x[tr], cv_y[tr], cv_x[va], h["z"], 0.1)
            ref.append(driver.nlpd(cv_y[va], m_, v_))
        assert np.max(np.abs(np.array(h["cv"]["fold_nlpds"]) - np.array(ref))) < 1e-7
        assert abs(h["cv"]["mean_nlpd"] - float(np.mean(ref))) < 1e-7


def test_generate_quantum_gp_data_dot_product_matches_numpy_cholesky(d):
    """generate_quantum_gp_data with the dot-product outer kernel (rank <= 3q + 1: K + 1e-6 I is positive definite only through
    the 1e-6) against NumPy: the same host draws, Y = chol(K + 1e-6 I) z + noise with the oracle's K.

    Tolerance from the conditioning: the two Grams and the two factorisations differ by backward errors of order n eps |A|_2,
    and the Cholesky factor's condition number is typically sqrt(kappa_2(A)) (Chang, Paige & Stewart 1996), so
    |dY|_inf <= n eps sqrt(kappa_2(A)) |L|_2 |z|_inf, with |L|_2 = sqrt(|A|_2).  Here kappa_2(A) ~ 3.5e9 and the bound is ~6e-6
    against |Y| ~ 4."""
    from oracle import qkernels
    n, dd, q, layers = 2048, 2, 3, 1
    X, Y, truth = d.generate_quantum_gp_data(n, dd, q, layers, (-2.0, 2.0), 0.1, True, None, "yz_cx", "projected", "XYZ",
                                             "dotproduct", None, None, data_seed=7, param_seed=42, lean=False)
    enc = qkernels.EncodingCircuit("yz_cx", q, dd, layers)
    np.random.seed(42)
    truth_ref = np.round(np.random.uniform(0, np.pi, enc.num_parameters), 4)
    np.random.seed(7)
    X_ref = np.random.uniform(-2.0, 2.0, size=(n, dd))
    assert np.array_equal(truth, truth_ref) and np.array_equal(X, X_ref)
    F = enc.features(X_ref, truth_ref)
    A = sk.DotProduct()(F, F) + 1e-6 * np.eye(n)
    z = np.random.normal(0, 1, n)
    Y_ref = np.linalg.cholesky(A) @ z
    Y_ref += np.random.normal(0, 0.1, n)
    ev = np.linalg.eigvalsh(A)
    kappa = ev[-1] / ev[0]
    tol = n * np.finfo(np.float64).eps * np.sqrt(kappa) * np.sqrt(ev[-1]) * np.abs(z).max()
    assert 1e8 < kappa < 1e11 and tol < 1e-4
    assert np.max(np.abs(Y - Y_ref)) <= tol
