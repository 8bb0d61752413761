"""GPU tests of the analytic NLL gradient (AgentEngine(gradient="analytic"), dqgp_grad_projected_analytic) for every outer kernel
of the projected kernel: the C ABI against differences of scikit-learn's kernels, NaN propagation, the engine against the oracle's
NLL on the Cholesky and the LU rung, and the CUDA-graph replays of RiemannianAgent and AdmmEngine in this mode."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
sk = pytest.importorskip("sklearn.gaussian_process.kernels")

# (outer id name, ABI hyper-parameters, the scikit-learn kernel with the same hyper-parameters)
CASES = [
    ("gaussian", [1.0], lambda: sk.RBF(length_scale=1.0 / np.sqrt(2.0))),
    ("gaussian", [0.6], lambda: sk.RBF(length_scale=1.0 / np.sqrt(1.2))),
    ("matern", [1.0], lambda: sk.Matern(nu=1.5)),
    ("matern", [0.7], lambda: sk.Matern(length_scale=0.7, nu=1.5)),
    ("expsinesquared", [1.0, 1.0], lambda: sk.ExpSineSquared()),
    ("expsinesquared", [0.8, 1.3], lambda: sk.ExpSineSquared(length_scale=0.8, periodicity=1.3)),
    ("rationalquadratic", [1.0, 1.0], lambda: sk.RationalQuadratic()),
    ("rationalquadratic", [0.7, 2.5], lambda: sk.RationalQuadratic(length_scale=0.7, alpha=2.5)),
    ("rationalquadratic", [0.7, 1.0], lambda: sk.RationalQuadratic(length_scale=0.7, alpha=1.0)),
    ("dotproduct", [1.0], lambda: sk.DotProduct()),
    ("dotproduct", [0.3], lambda: sk.DotProduct(sigma_0=0.3)),
    ("dotproduct", [0.0], lambda: sk.PairwiseKernel(metric="linear")),
]
CASE_IDS = [f"{name}-{'-'.join(str(v) for v in hyp)}" for name, hyp, _ in CASES]


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


def _inputs(rng, n, m, P):
    """Features in [-1, 1], a Jacobian, a random symmetric A^-1 and alpha; sample 3 duplicates sample 0 (features and Jacobian)."""
    F = rng.uniform(-1, 1, (n, m))
    J = rng.standard_normal((P, n, m))
    if n > 3:
        F[3], J[:, 3] = F[0], J[:, 0]
    A = rng.standard_normal((n, n))
    return F, J, A + A.T, rng.standard_normal(n)


def _device_gradient(d, outer, hyp, Ainv, alpha, F, J):
    """dqgp_grad_projected_analytic with ld = n + 3; the padding columns of A^-1 hold NaN, so a read past n would show."""
    from dqgp_b200 import _lib
    lib = d.load()
    n, m = F.shape
    P = J.shape[0]
    ld = n + 3
    A = np.full((n, ld), np.nan)
    A[:, :n] = Ainv
    dA, dal, dF, dJ = (d.kernels.dev_f64(v) for v in (A, alpha, F, J))
    work = torch.empty(lib.dqgp_grad_analytic_workspace_bytes(n, m) // 8 + 1, dtype=torch.float64, device="cuda")
    grad = torch.full((P,), -7.0, dtype=torch.float64, device="cuda")
    rc = lib.dqgp_grad_projected_analytic(_lib.OUTER_KERNELS[outer], _lib.hyp_array(hyp), dA.data_ptr(), ld, dal.data_ptr(),
                                          dF.data_ptr(), dJ.data_ptr(), n, m, P, grad.data_ptr(), work.data_ptr(), _sp())
    assert rc == 0, lib.dqgp_last_error()
    torch.cuda.synchronize()
    return grad.cpu().numpy()


def _sklearn_gradient(kernel, F, J, B, t=1e-4):
    """1/2 sum(B o dK_i), dK_i the 4-point difference of the scikit-learn kernel along J_i: independent of the device formulas."""
    out = []
    for Ji in J:
        k = lambda s: kernel(F + s * Ji)
        dK = (-k(2 * t) + 8 * k(t) - 8 * k(-t) + k(-2 * t)) / (12 * t)
        out.append(0.5 * np.sum(B * dK))
    return np.array(out)


@pytest.mark.parametrize("m", [9, 24, 36])
@pytest.mark.parametrize("case", range(len(CASES)), ids=CASE_IDS)
def test_abi_matches_scikit_learn_differences(d, case, m):
    """Every outer id at its default and a non-default hyper-parameter, ragged n, ld > n, duplicate samples: the gradient equals
    differences of scikit-learn's kernel to 1e-9 of its largest entry, and a second call gives the same bits."""
    outer, hyp, kernel = CASES[case]
    rng = np.random.default_rng(100 * case + m)
    for n in [1, 63, 65, 200]:
        F, J, Ainv, alpha = _inputs(rng, n, m, 3)
        ref = _sklearn_gradient(kernel(), F, J, Ainv - np.outer(alpha, alpha))
        got = _device_gradient(d, outer, hyp, Ainv, alpha, F, J)
        assert np.all(np.abs(got - ref) <= 1e-9 * np.abs(ref).max()), (n, got, ref)
        assert np.array_equal(got, _device_gradient(d, outer, hyp, Ainv, alpha, F, J))


@pytest.mark.parametrize("outer,hyp", [("matern", [1.0]), ("expsinesquared", [1.0, 1.0]), ("rationalquadratic", [1.0, 1.0]),
                                       ("rationalquadratic", [0.7, 2.5]), ("dotproduct", [1.0])])
def test_nan_feature_gives_a_nan_gradient(d, outer, hyp):
    """A NaN feature (arccos outside [-1, 1]) reaches every entry of the gradient, as in NumPy: no guard turns it into a number."""
    rng = np.random.default_rng(7)
    F, J, Ainv, alpha = _inputs(rng, 70, 9, 4)
    F[5, 4] = np.nan
    assert np.all(np.isnan(_device_gradient(d, outer, hyp, Ainv, alpha, F, J)))


def _oracle_nll(x, y, q, dd, layers, enc, outer, p):
    """(sign of det A, 1/2 log|det A| + 1/2 y^T A^-1 y + n/2 log 2 pi) with A = K + 0.01 I from the oracle's kernel.  Its derivative
    is 1/2 sum (A^-1 - alpha alpha^T) o dA whether or not A is positive definite."""
    from oracle import qkernels
    qk = qkernels.create_quantum_kernel(q, dd, layers, enc, "projected", "XYZ", outer)
    qk.assign_parameters(p)
    a = qk.evaluate(x, x) + 0.01 * np.eye(len(y))
    sign, logabs = np.linalg.slogdet(a)
    return sign, 0.5 * logabs + 0.5 * y @ np.linalg.solve(a, y) + 0.5 * len(y) * np.log(2 * np.pi)


def _check_against_oracle_nll(eng, x, y, q, dd, layers, enc, outer, z):
    sign, ref_nll = _oracle_nll(x, y, q, dd, layers, enc, outer, z)
    nll = float(eng.d_nll[3].item())
    if sign > 0:
        assert abs(nll - ref_nll) < 1e-8 * abs(ref_nll)
    else:
        assert np.isnan(nll)                  # the reference takes the log of a non-positive determinant
    grad = eng.d_grad.cpu().numpy()
    h = 1e-5
    for i in range(0, len(z), max(1, len(z) // 5)):
        e = np.zeros_like(z)
        e[i] = h
        ref = (_oracle_nll(x, y, q, dd, layers, enc, outer, z + e)[1] - _oracle_nll(x, y, q, dd, layers, enc, outer, z - e)[1]) / (2 * h)
        assert abs(grad[i] - ref) < 2e-5 * max(1.0, abs(ref)), (i, grad[i], ref)


@pytest.mark.parametrize("outer", ["matern", "expsinesquared", "rationalquadratic", "dotproduct", "pairwisekernel"])
@pytest.mark.parametrize("enc,q,dd,layers,n", [("kyriienko", 3, 6, 1, 128), ("yz_cx", 3, 2, 2, 150), ("chebyshev", 3, 2, 1, 130)])
def test_engine_gradient_is_the_derivative_of_the_oracle_nll(d, sklearn_oracle, outer, enc, q, dd, layers, n):
    """AgentEngine(gradient="analytic", training_ignores_outer_kernel=False): the NLL equals the oracle's, and the gradient equals
    central differences of the oracle's NLL with that outer kernel.  ExpSineSquared's Gram is indefinite here: its step takes
    the LU rung, as AgentEngine.step_fallback does."""
    x, y = d.synthetic_dataset(n, dd, enc)
    z = np.round(np.random.RandomState(5).uniform(0.2, 2.9, d.EncodingCircuit(enc, q, dd, layers).num_parameters), 4)
    eng = d.AgentEngine(x, y, encoding_type=enc, kernel_type="projected", num_qubits=q, num_layers=layers, noise_std=0.1, rho=100.0,
                        L=100.0, outer_kernel=outer, training_ignores_outer_kernel=False, gradient="analytic")
    eng.simulate(d.kernels.dev_f64(z)); eng.gram(); eng.factor()
    torch.cuda.synchronize()
    if int(eng.d_info.item()) != 0:
        assert outer == "expsinesquared"
        eng.gram(full=True); eng.factor_lu()
    eng.gradient()
    torch.cuda.synchronize()
    _check_against_oracle_nll(eng, x, y, q, dd, layers, enc, outer, z)


def test_lu_rung_gradient_is_the_derivative_of_log_abs_det(d):
    """The inputs of test_agent_step_walks_the_lu_rung_when_cholesky_fails (ExpSineSquared honoured, Cholesky fails): after
    step_fallback the analytic gradient equals differences of 1/2 log|det A| + 1/2 y^T A^-1 y computed with slogdet."""
    x, y = d.synthetic_dataset(97, 4, "hubregtsen", seed=5)
    rs = np.random.RandomState(8)
    z, psi = np.round(rs.rand(12) * np.pi, 4), np.round(rs.rand(12), 4)
    eng = d.AgentEngine(x, y, encoding_type="hubregtsen", kernel_type="projected", num_qubits=3, num_layers=2, noise_std=0.1,
                        rho=100.0, L=100.0, outer_kernel="expsinesquared", training_ignores_outer_kernel=False, gradient="analytic")
    dz, dpsi = d.kernels.dev_f64(z), d.kernels.dev_f64(psi)
    theta, psi_out = torch.empty_like(dz), torch.empty_like(dz)
    eng.step(dz, dpsi, theta, psi_out)
    torch.cuda.synchronize()
    assert int(eng.d_info.item()) != 0
    eng.step_fallback(dz, dpsi, theta, psi_out)
    torch.cuda.synchronize()
    assert eng.used_lu_fallback
    _check_against_oracle_nll(eng, x, y, 3, 4, 2, "hubregtsen", "expsinesquared", np.mod(z, np.pi))


def test_riemannian_agent_graph_replay_equals_eager(d):
    """RiemannianAgent(outer_kernel="matern", training_ignores_outer_kernel=False, gradient="analytic"): the second call, which
    replays the step as a CUDA graph, returns exactly what the first (eager) call returned on the same inputs, and theta / psi
    follow from the rounded gradient by the reference's local update."""
    from oracle import agent_step, torus
    x, y = d.synthetic_dataset(140, 2, "yz_cx")
    rs = np.random.RandomState(11)
    P = d.EncodingCircuit("yz_cx", 4, 2, 2).num_parameters
    z, psi = np.round(rs.uniform(0.2, 2.9, P), 4), np.round(rs.rand(P), 4)
    ag = d.RiemannianAgent("analytic_matern", x, y, 4, 0.1, 100.0, 100.0, use_parameter_shift=True, num_layers=2,
                           encoding_type="yz_cx", kernel_type="projected", outer_kernel="matern", training_ignores_outer_kernel=False,
                           gradient="analytic")
    eager = ag.train_and_update(z, psi)
    g_eager = ag.last_gradient.copy()
    assert ag._engine()._graph is None
    replayed = ag.train_and_update(z, psi)
    assert ag._engine()._graph is not None
    for a, b in zip(eager[:3], replayed[:3]):
        assert np.array_equal(a, b)
    assert np.array_equal(g_eager, ag.last_gradient)
    th_ref, ps_ref = agent_step.local_update(torus.wrap(z), np.round(g_eager, 4), psi, 100.0, 100.0)
    assert np.max(np.abs(replayed[0] - th_ref)) < 1e-12 and np.max(np.abs(replayed[1] - ps_ref)) < 1e-9


def test_admm_engine_graph_replay_equals_eager_iterations(d):
    """AdmmEngine.capture()/replay() walks the same trajectory as eager iteration() calls with the analytic gradient and the
    Matern outer kernel honoured in training."""
    x, y = d.synthetic_dataset(4 * 150, 2, "chebyshev")
    shards = [(x[a * 150:(a + 1) * 150], y[a * 150:(a + 1) * 150]) for a in range(4)]
    rs = np.random.RandomState(42)
    theta0, psi0 = np.round(rs.rand(4, 12), 4), np.round(rs.rand(4, 12), 4)
    kw = dict(rho=100.0, L=100.0, encoding_type="chebyshev", kernel_type="projected", num_qubits=3, num_layers=1, noise_std=0.1,
              outer_kernel="matern", training_ignores_outer_kernel=False, gradient="analytic")
    eager = d.AdmmEngine(shards, theta0, psi0, **kw)
    for _ in range(4):
        eager.iteration()
    graph = d.AdmmEngine(shards, theta0, psi0, **kw)
    graph.capture()
    for _ in range(4):
        graph.replay()
    for a, b in zip(eager.state(), graph.state()):
        assert np.array_equal(a, b)
    assert all(ag.gradient_mode == "analytic" for ag in graph.agents)
