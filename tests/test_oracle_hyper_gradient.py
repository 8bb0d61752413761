"""The derivative formulas of the outer-kernel hyper-parameter gradient (dqgp_grad_outer_hyperparameters), in NumPy, against
scikit-learn's own ``eval_gradient=True`` (no device needed).

The device contracts B = A^-1 - alpha alpha^T with dK/dh, h the values exactly as they appear in h_hyp: gamma for the Gaussian
(scikit-learn's RBF has length_scale = 1 / sqrt(2 gamma)), length_scale, periodicity, alpha and sigma_0 for the others.
scikit-learn returns dK/dlog(theta), one column per entry of ``kernel.hyperparameters`` (sorted by name)."""
import numpy as np
import pytest
from scipy.spatial.distance import cdist

sk = pytest.importorskip("sklearn.gaussian_process.kernels")


def hyper_derivatives(outer, hyp, F):
    """dK/dh for every entry of hyp (the table of include/dqgp.h), d = |f_j - f_k|, s = d^2."""
    s = cdist(F, F, metric="sqeuclidean")
    d = np.sqrt(s)
    if outer == "gaussian":
        (g,) = hyp
        K = np.exp(-g * s)
        return [-s * K]
    if outer == "matern":
        (l,) = hyp
        k = np.sqrt(3.0) * d / l
        return [k * k * np.exp(-k) / l]
    if outer == "expsinesquared":
        l, p = hyp
        sn = np.sin(np.pi * d / p)
        K = np.exp(-2.0 * sn * sn / (l * l))
        return [4.0 * sn * sn / l ** 3 * K, 2.0 * np.pi * d / (l * l * p * p) * np.sin(2.0 * np.pi * d / p) * K]
    if outer == "rationalquadratic":
        l, a = hyp
        u = s / (2.0 * a * l * l)
        K = np.exp(-a * np.log1p(u))
        return [2.0 * a * u * K / (l * (1.0 + u)), K * (u / (1.0 + u) - np.log1p(u))]
    if outer == "dotproduct":
        (s0,) = hyp
        return [np.full_like(s, 2.0 * s0)]
    raise ValueError(outer)


# (outer id name, h_hyp, the scikit-learn kernel, the name of each h_hyp entry in kernel.hyperparameters, h -> theta)
CASES = [
    ("gaussian", [1.0], lambda: sk.RBF(length_scale=1.0 / np.sqrt(2.0)), ["length_scale"]),
    ("gaussian", [0.6], lambda: sk.RBF(length_scale=1.0 / np.sqrt(1.2)), ["length_scale"]),
    ("matern", [1.0], lambda: sk.Matern(nu=1.5), ["length_scale"]),
    ("matern", [0.7], lambda: sk.Matern(length_scale=0.7, nu=1.5), ["length_scale"]),
    ("expsinesquared", [1.0, 1.0], lambda: sk.ExpSineSquared(), ["length_scale", "periodicity"]),
    ("expsinesquared", [0.8, 1.3], lambda: sk.ExpSineSquared(length_scale=0.8, periodicity=1.3), ["length_scale", "periodicity"]),
    ("rationalquadratic", [1.0, 1.0], lambda: sk.RationalQuadratic(), ["length_scale", "alpha"]),
    ("rationalquadratic", [0.7, 2.5], lambda: sk.RationalQuadratic(length_scale=0.7, alpha=2.5), ["length_scale", "alpha"]),
    ("dotproduct", [1.0], lambda: sk.DotProduct(), ["sigma_0"]),
    ("dotproduct", [0.3], lambda: sk.DotProduct(sigma_0=0.3), ["sigma_0"]),
]
CASE_IDS = [f"{name}-{'-'.join(str(v) for v in hyp)}" for name, hyp, _, _ in CASES]


def sklearn_hyper_derivatives(outer, hyp, kernel, names, F):
    """dK/dh from scikit-learn's dK/dlog(theta): columns matched to h_hyp by name, then divided by theta; the Gaussian's
    gamma = 1 / (2 l^2) gives dK/dgamma = -(dK/dlog l) / (2 gamma)."""
    _, G = kernel(F, eval_gradient=True)
    cols = {hp.name: i for i, hp in enumerate(hp for hp in kernel.hyperparameters if not hp.fixed)}
    theta = dict(zip((hp.name for hp in kernel.hyperparameters if not hp.fixed), np.exp(kernel.theta)))
    if outer == "gaussian":
        return [-G[:, :, cols["length_scale"]] / (2.0 * hyp[0])]
    return [G[:, :, cols[nm]] / theta[nm] for nm in names]


def _points(seed):
    rng = np.random.default_rng(seed)
    F = rng.uniform(-1, 1, (30, 6))
    F[7] = F[2]                                  # a duplicate sample: s = 0 off the diagonal
    return F


@pytest.mark.parametrize("case", range(len(CASES)), ids=CASE_IDS)
def test_derivatives_match_scikit_learn_eval_gradient(case):
    outer, hyp, kernel, names = CASES[case]
    F = _points(case)
    ours = hyper_derivatives(outer, hyp, F)
    ref = sklearn_hyper_derivatives(outer, hyp, kernel(), names, F)
    assert len(ours) == len(ref) == len(hyp)
    for a, b in zip(ours, ref):
        assert np.allclose(a, b, rtol=1e-13, atol=1e-15 * np.abs(b).max()), np.abs(a - b).max()


@pytest.mark.parametrize("case", [c for c in range(len(CASES)) if CASES[c][0] != "dotproduct"], ids=lambda c: CASE_IDS[c])
def test_stationary_derivatives_vanish_at_zero_distance(case):
    """The diagonal and the duplicate pair (s = 0) have exactly zero derivative for every stationary outer kernel."""
    outer, hyp, _, _ = CASES[case]
    F = _points(case)
    for D in hyper_derivatives(outer, hyp, F):
        assert np.all(np.diagonal(D) == 0.0) and D[7, 2] == 0.0 and D[2, 7] == 0.0


def test_lower_triangle_weighting_is_the_full_contraction():
    """The device sums j > k with weight 2 and j = k with weight 1 and never reads j < k: for a symmetric B and dK that is
    the full sum of B o dK."""
    rng = np.random.default_rng(3)
    F = _points(11)
    B = rng.standard_normal((30, 30))
    B = B + B.T
    for outer, hyp, _, _ in CASES:
        for D in hyper_derivatives(outer, hyp, F):
            W = np.tril(np.full((30, 30), 2.0), -1) + np.eye(30)
            assert np.isclose(np.sum(W * B * D), np.sum(B * D), rtol=1e-13, atol=1e-13)


def test_noise_derivative_is_sigma_trace_b():
    """dNLL/dsigma = sigma tr(A^-1 - alpha alpha^T) for A = K + sigma^2 I, against a central difference of the NLL."""
    rng = np.random.default_rng(4)
    F = _points(4)
    K = sk.RBF(0.8)(F)
    y = rng.standard_normal(30)

    def nll(sig):
        A = K + sig * sig * np.eye(30)
        return 0.5 * np.linalg.slogdet(A)[1] + 0.5 * y @ np.linalg.solve(A, y)

    sig = 0.3
    A = K + sig * sig * np.eye(30)
    Ainv = np.linalg.inv(A)
    al = Ainv @ y
    got = sig * (np.trace(Ainv) - al @ al)
    h = 1e-6
    assert np.isclose(got, (nll(sig + h) - nll(sig - h)) / (2 * h), rtol=1e-7)
