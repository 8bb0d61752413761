"""GPU tests of the NLL gradient with respect to the outer kernel's hyper-parameters and the noise level
(dqgp_grad_outer_hyperparameters, dqgp_grad_noise_std, AgentEngine(hyper_gradient=True)): the C ABI against scikit-learn's
eval_gradient, NaN propagation, the engine against central differences of a reference NLL (Cholesky and LU rung, both gradient
modes), CUDA-graph replays of AdmmEngine, and argument validation."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
sk = pytest.importorskip("sklearn.gaussian_process.kernels")

from test_gpu_analytic_outer_kernels import CASE_IDS, CASES  # noqa: E402
from test_oracle_hyper_gradient import sklearn_hyper_derivatives  # noqa: E402

# scikit-learn's name of each h_hyp entry
NAMES = {"gaussian": ["length_scale"], "matern": ["length_scale"], "expsinesquared": ["length_scale", "periodicity"],
         "rationalquadratic": ["length_scale", "alpha"], "dotproduct": ["sigma_0"]}
# non-default hyper-parameters in the reference's format, and the scikit-learn kernel they describe
PARAMS = {
    "gaussian": ({"gamma": 0.6}, lambda p: sk.RBF(length_scale=1.0 / np.sqrt(2.0 * p["gamma"]))),
    "matern": ({"length_scale": 0.7}, lambda p: sk.Matern(length_scale=p["length_scale"], nu=1.5)),
    "expsinesquared": ({"length_scale": 0.8, "periodicity": 1.3},
                       lambda p: sk.ExpSineSquared(length_scale=p["length_scale"], periodicity=p["periodicity"])),
    "rationalquadratic": ({"length_scale": 0.7, "alpha": 2.5}, lambda p: sk.RationalQuadratic(length_scale=p["length_scale"], alpha=p["alpha"])),
    "dotproduct": ({"sigma_0": 0.3}, lambda p: sk.DotProduct(sigma_0=p["sigma_0"])),
    "pairwisekernel": ({"metric": "linear"}, lambda p: sk.PairwiseKernel(metric="linear")),
}


@pytest.fixture(scope="module")
def d():
    import dqgp_b200
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")
    return dqgp_b200


def _sp():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _inputs(rng, n, m):
    """Features in [-1, 1] (sample 3 duplicates sample 0), a random symmetric A^-1 and alpha."""
    F = rng.uniform(-1, 1, (n, m))
    if n > 3:
        F[3] = F[0]
    A = rng.standard_normal((n, n))
    return F, A + A.T, rng.standard_normal(n)


def _device_hyper_gradient(d, outer, hyp, Ainv, alpha, F, noise_std=0.1):
    """Both entry points with ld = n + 3: the padding columns and the strict upper triangle of A^-1 hold NaN, so a read of any
    entry with j < k would show.  Returns (dNLL/dh, dNLL/dsigma)."""
    from dqgp_b200 import _lib
    lib = d.load()
    n, m = F.shape
    ld = n + 3
    A = np.full((n, ld), np.nan)
    A[:, :n] = np.where(np.tril(np.ones((n, n), dtype=bool)), Ainv, np.nan)
    dA, dal, dF = (d.kernels.dev_f64(v) for v in (A, alpha, F))
    work = torch.empty(lib.dqgp_grad_outer_hyperparameters_workspace_bytes(n) // 8 + 1, dtype=torch.float64, device="cuda")
    grad = torch.full((len(hyp) + 1,), -7.0, dtype=torch.float64, device="cuda")
    rc = lib.dqgp_grad_outer_hyperparameters(_lib.OUTER_KERNELS[outer], _lib.hyp_array(hyp), dA.data_ptr(), ld, dal.data_ptr(),
                                             dF.data_ptr(), n, m, grad.data_ptr(), work.data_ptr(), _sp())
    assert rc == 0, lib.dqgp_last_error()
    rc = lib.dqgp_grad_noise_std(dA.data_ptr(), ld, dal.data_ptr(), n, noise_std, grad[len(hyp):].data_ptr(), _sp())
    assert rc == 0, lib.dqgp_last_error()
    torch.cuda.synchronize()
    g = grad.cpu().numpy()
    return g[:len(hyp)], g[len(hyp)]


@pytest.mark.parametrize("m", [9, 24, 36])
@pytest.mark.parametrize("case", range(len(CASES)), ids=CASE_IDS)
def test_abi_matches_scikit_learn_eval_gradient(d, case, m):
    """Every outer id at its default and a non-default hyper-parameter, ragged n, ld > n, NaN above the diagonal, a duplicate
    sample: the result equals 1/2 sum B o dK/dh from scikit-learn's eval_gradient to 1e-9 of 1/2 sum |B o dK/dh|, the noise entry
    equals sigma tr(B), and a second call gives the same bits."""
    outer, hyp, kernel = CASES[case]
    rng = np.random.default_rng(100 * case + m + 1)
    for n in [1, 63, 65, 200]:
        F, Ainv, alpha = _inputs(rng, n, m)
        B = Ainv - np.outer(alpha, alpha)
        if outer == "dotproduct" and hyp == [0.0]:
            dK = [np.zeros((n, n))]                      # PairwiseKernel(metric="linear") has no sigma_0: 2 sigma_0 = 0
        else:
            dK = sklearn_hyper_derivatives(outer, hyp, kernel(), NAMES[outer], F)
        ref = np.array([0.5 * np.sum(B * D) for D in dK])
        scale = np.array([0.5 * np.sum(np.abs(B * D)) for D in dK])
        got, noise = _device_hyper_gradient(d, outer, hyp, Ainv, alpha, F)
        assert np.all(np.abs(got - ref) <= 1e-9 * scale), (n, got, ref)
        assert abs(noise - 0.1 * np.trace(B)) <= 1e-12 * np.sum(np.abs(np.diagonal(B))) * 0.1, (n, noise)
        again = _device_hyper_gradient(d, outer, hyp, Ainv, alpha, F)
        assert np.array_equal(got, again[0]) and noise == again[1]


@pytest.mark.parametrize("outer,hyp", [("gaussian", [0.6]), ("matern", [1.0]), ("expsinesquared", [0.8, 1.3]),
                                       ("rationalquadratic", [1.0, 1.0]), ("rationalquadratic", [0.7, 2.5])])
def test_nan_feature_gives_a_nan_hyper_gradient(d, outer, hyp):
    """A NaN feature (arccos outside [-1, 1]) reaches every hyper-parameter entry of every stationary outer kernel."""
    rng = np.random.default_rng(7)
    F, Ainv, alpha = _inputs(rng, 70, 9)
    F[5, 4] = np.nan
    got, _ = _device_hyper_gradient(d, outer, hyp, Ainv, alpha, F)
    assert np.all(np.isnan(got))


def _reference_nll(F, y, kernel, noise_std):
    """1/2 log|det A| + 1/2 y^T A^-1 y + n/2 log 2 pi, A = K + sigma^2 I from scikit-learn's kernel: its derivative is
    1/2 sum B o dA whether or not A is positive definite.  Returns (sign of det A, NLL)."""
    a = kernel(F) + noise_std ** 2 * np.eye(len(y))
    sign, logabs = np.linalg.slogdet(a)
    return sign, 0.5 * logabs + 0.5 * y @ np.linalg.solve(a, y) + 0.5 * len(y) * np.log(2 * np.pi)


def _engine_step(d, x, y, enc, q, layers, outer, params, mode, z):
    """AgentEngine phases on z; a failed Cholesky walks the LU rung as step_fallback does."""
    eng = d.AgentEngine(x, y, encoding_type=enc, kernel_type="projected", num_qubits=q, num_layers=layers, noise_std=0.1, rho=100.0,
                        L=100.0, outer_kernel=outer, training_ignores_outer_kernel=False, outer_kernel_params=params,
                        gradient=mode, hyper_gradient=True)
    eng.simulate(d.kernels.dev_f64(z)); eng.gram(); eng.factor()
    torch.cuda.synchronize()
    if int(eng.d_info.item()) != 0:
        eng.gram(full=True); eng.factor_lu()
    eng.gradient()
    return eng, eng.hyper_gradient()


def _check_against_reference_nll(eng, got, F, y, outer, params):
    """The engine's NLL equals the reference's to 1e-8, and every hyper entry and noise_std equal central differences of it."""
    make = PARAMS[outer][1]
    sign, ref_nll = _reference_nll(F, y, make(params), 0.1)
    nll = float(eng.d_nll[3].item())
    if sign > 0:
        assert abs(nll - ref_nll) < 1e-8 * abs(ref_nll)
    else:
        assert np.isnan(nll)                  # the log of a non-positive determinant, as the reference takes it
    assert list(got) == eng.hyper_names + ["noise_std"]
    for name in eng.hyper_names:
        ref = _central_difference(lambda t: _reference_nll(F, y, make(dict(params, **{name: params[name] + t})), 0.1)[1])
        assert abs(got[name] - ref) < 2e-5 * max(1.0, abs(ref)), (name, got[name], ref)
    ref = _central_difference(lambda t: _reference_nll(F, y, make(params), 0.1 + t)[1])
    assert abs(got["noise_std"] - ref) < 2e-5 * max(1.0, abs(ref)), ("noise_std", got["noise_std"], ref)


def _central_difference(f, h=1e-5):
    """4-point central difference: near-singular A (ExpSineSquared) curves the NLL enough that the 2-point rule's h^2 term
    reaches 1e-4 relative at h = 1e-5."""
    return (-f(2 * h) + 8 * f(h) - 8 * f(-h) + f(-2 * h)) / (12 * h)


@pytest.mark.parametrize("outer", list(PARAMS))
@pytest.mark.parametrize("enc,q,dd,layers,n", [("yz_cx", 3, 2, 2, 150), ("chebyshev", 3, 2, 1, 130)])
def test_engine_hyper_gradient_is_the_derivative_of_the_reference_nll(d, outer, enc, q, dd, layers, n):
    """AgentEngine(training_ignores_outer_kernel=False, outer_kernel_params=non-default, hyper_gradient=True) in both gradient
    modes: the NLL equals the one built from the oracle's features and scikit-learn's kernel at those values, every entry equals
    central differences of it, and the two modes agree to 1e-12."""
    from oracle import qkernels
    x, y = d.synthetic_dataset(n, dd, enc)
    z = np.round(np.random.RandomState(5).uniform(0.2, 2.9, d.EncodingCircuit(enc, q, dd, layers).num_parameters), 4)
    F = qkernels.EncodingCircuit(enc, q, dd, layers).features(x, z)
    params = PARAMS[outer][0]
    results = {}
    for mode in ("central_difference", "analytic"):
        eng, got = _engine_step(d, x, y, enc, q, layers, outer, params, mode, z)
        _check_against_reference_nll(eng, got, F, y, outer, params)
        results[mode] = got
    for name, v in results["central_difference"].items():
        assert abs(v - results["analytic"][name]) <= 1e-12 * max(1.0, abs(v)), (name, v, results["analytic"][name])


@pytest.mark.parametrize("mode", ["central_difference", "analytic"])
def test_lu_rung_hyper_gradient_is_the_derivative_of_log_abs_det(d, mode):
    """The inputs of test_lu_rung_gradient_is_the_derivative_of_log_abs_det (ExpSineSquared honoured, Cholesky fails): after
    step_fallback the hyper-gradient equals differences of the slogdet-based NLL."""
    from oracle import qkernels
    x, y = d.synthetic_dataset(97, 4, "hubregtsen", seed=5)
    rs = np.random.RandomState(8)
    z, psi = np.round(rs.rand(12) * np.pi, 4), np.round(rs.rand(12), 4)
    params = {"length_scale": 1.0, "periodicity": 1.0}
    eng = d.AgentEngine(x, y, encoding_type="hubregtsen", kernel_type="projected", num_qubits=3, num_layers=2, noise_std=0.1,
                        rho=100.0, L=100.0, outer_kernel="expsinesquared", training_ignores_outer_kernel=False,
                        outer_kernel_params=params, gradient=mode, hyper_gradient=True)
    dz, dpsi = d.kernels.dev_f64(z), d.kernels.dev_f64(psi)
    theta, psi_out = torch.empty_like(dz), torch.empty_like(dz)
    eng.step(dz, dpsi, theta, psi_out)
    torch.cuda.synchronize()
    assert int(eng.d_info.item()) != 0
    eng.step_fallback(dz, dpsi, theta, psi_out)
    assert eng.used_lu_fallback
    F = qkernels.EncodingCircuit("hubregtsen", 3, 4, 2).features(x, np.mod(z, np.pi))
    _check_against_reference_nll(eng, eng.hyper_gradient(), F, y, "expsinesquared", params)


@pytest.mark.parametrize("mode", ["central_difference", "analytic"])
def test_admm_engine_graph_replay_equals_eager_iterations(d, mode):
    """AdmmEngine.capture()/replay() with hyper_gradient=True gives the same state() and hyper_gradients() bits as eager
    iteration() calls."""
    x, y = d.synthetic_dataset(4 * 150, 2, "chebyshev")
    shards = [(x[a * 150:(a + 1) * 150], y[a * 150:(a + 1) * 150]) for a in range(4)]
    rs = np.random.RandomState(42)
    theta0, psi0 = np.round(rs.rand(4, 12), 4), np.round(rs.rand(4, 12), 4)
    kw = dict(rho=100.0, L=100.0, encoding_type="chebyshev", kernel_type="projected", num_qubits=3, num_layers=1, noise_std=0.1,
              outer_kernel="rationalquadratic", training_ignores_outer_kernel=False,
              outer_kernel_params={"length_scale": 0.7, "alpha": 2.5}, gradient=mode, hyper_gradient=True)
    eager = d.AdmmEngine(shards, theta0, psi0, **kw)
    for _ in range(4):
        eager.iteration()
    graph = d.AdmmEngine(shards, theta0, psi0, **kw)
    graph.capture()
    for _ in range(4):
        graph.replay()
    for a, b in zip(eager.state(), graph.state()):
        assert np.array_equal(a, b)
    he, hg = eager.hyper_gradients(), graph.hyper_gradients()
    assert he.shape == (4, 3) and np.all(np.isfinite(he))
    assert np.array_equal(he, hg)


def test_validation(d):
    """outer_kernel_params where the training kernel ignores the outer kernel raises ValueError; a length scale <= 0 raises
    DqgpError; the fidelity kernel returns only noise_std, equal to sigma tr(A^-1 - alpha alpha^T); the flag adds its launches."""
    from dqgp_b200 import _lib
    x, y = d.synthetic_dataset(80, 2, "yz_cx")
    kw = dict(encoding_type="yz_cx", num_qubits=3, num_layers=1, noise_std=0.1, rho=100.0, L=100.0)
    with pytest.raises(ValueError):
        d.AgentEngine(x, y, kernel_type="projected", outer_kernel="matern", outer_kernel_params={"length_scale": 0.7}, **kw)
    with pytest.raises(ValueError):
        d.AgentEngine(x, y, kernel_type="fidelity", training_ignores_outer_kernel=False, outer_kernel_params={"gamma": 0.5}, **kw)
    P = d.EncodingCircuit("yz_cx", 3, 2, 1).num_parameters
    z = d.kernels.dev_f64(np.linspace(0.3, 2.5, P))
    out = [torch.zeros_like(z) for _ in range(3)]
    bad = d.AgentEngine(x, y, kernel_type="projected", outer_kernel="matern", training_ignores_outer_kernel=False,
                        outer_kernel_params={"length_scale": 0.0}, hyper_gradient=True, **kw)
    with pytest.raises(_lib.DqgpError):
        bad.step(z, out[0], out[1], out[2])
    F = d.kernels.dev_f64(np.zeros((4, 9)))
    A = d.kernels.dev_f64(np.eye(4))
    work = torch.empty(16, dtype=torch.float64, device="cuda")
    lib = d.load()
    assert lib.dqgp_grad_outer_hyperparameters(1, _lib.hyp_array([-1.0]), A.data_ptr(), 4, F.data_ptr(), F.data_ptr(), 4, 9,
                                               work.data_ptr(), work.data_ptr(), _sp()) < 0
    assert lib.dqgp_grad_outer_hyperparameters(0, _lib.hyp_array([1.0]), A.data_ptr(), 4, F.data_ptr(), F.data_ptr(), 4, 37,
                                               work.data_ptr(), work.data_ptr(), _sp()) < 0
    fid = d.AgentEngine(x, y, kernel_type="fidelity", hyper_gradient=True, **kw)
    fid.step(z, out[0], out[1], out[2])
    got = fid.hyper_gradient()
    assert list(got) == ["noise_std"]
    B = fid.solver.inverse().diagonal() - fid.d_alpha * fid.d_alpha
    assert abs(got["noise_std"] - 0.1 * float(B.sum())) <= 1e-12 * 0.1 * float(B.abs().sum())
    plain = d.AgentEngine(x, y, kernel_type="fidelity", **kw)
    assert fid.launches_per_step() == plain.launches_per_step() + 1
    proj = dict(kernel_type="projected", outer_kernel="expsinesquared", training_ignores_outer_kernel=False, **kw)
    assert (d.AgentEngine(x, y, hyper_gradient=True, **proj).launches_per_step()
            == d.AgentEngine(x, y, **proj).launches_per_step() + 3)
