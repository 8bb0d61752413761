"""The reference for the RationalQuadratic, DotProduct and PairwiseKernel outer kernels (the rest of the reference's
--outer-kernel choices, main.py:1996-2013), and the host hyper-parameter mapping of the GPU path (no device needed).

squlearn maps these names to the scikit-learn kernel class with default hyper-parameters evaluated on (f(x), f(y))
(SURVEY A.4).  ``sklearn_outer_kernel_matrix`` is that mapping, with the installed classes; the GPU tests install it in place
of ``oracle.qkernels.outer_kernel_matrix`` (which covers the three outer kernels of the golden files) so that the oracle's
agent step, prediction and driver cover the new kernels unchanged."""
import math

import numpy as np
import pytest
from scipy.spatial.distance import cdist

from oracle import qkernels

sk = pytest.importorskip("sklearn.gaussian_process.kernels")

_ORACLE_OUTER_KERNEL_MATRIX = qkernels.outer_kernel_matrix

SKLEARN_OUTER = {
    "rationalquadratic": lambda p: sk.RationalQuadratic(length_scale=p.get("length_scale", 1.0), alpha=p.get("alpha", 1.0)),
    "dotproduct": lambda p: sk.DotProduct(sigma_0=p.get("sigma_0", 1.0)),
    "pairwisekernel": lambda p: sk.PairwiseKernel(gamma=p.get("gamma", 1.0), metric=p.get("metric", "linear")),
}


def sklearn_outer_kernel_matrix(name, f, g, **params):
    """outer_kernel_matrix with the three kernels above taken from scikit-learn (g=None: its symmetric call k(X)); every other
    name goes to the oracle's own outer_kernel_matrix."""
    if name in SKLEARN_OUTER:
        return SKLEARN_OUTER[name](params)(f, g)
    return _ORACLE_OUTER_KERNEL_MATRIX(name, f, g, **params)


@pytest.mark.parametrize("n1,n2,m", [(1, 1, 3), (24, 17, 24), (65, 63, 9), (40, 40, 36)])
def test_scikit_learn_defaults_are_the_documented_formulas(n1, n2, m):
    """The installed classes at their defaults compute the formulas the device kernels implement:
    RationalQuadratic 1 / (1 + |f-g|^2 / 2), DotProduct 1 + f.g, PairwiseKernel(metric="linear") f.g, with k(f, f) = 1,
    1 + |f|^2 and |f|^2."""
    rng = np.random.default_rng(n1 * 1000 + n2 + m)
    f, g = rng.uniform(-1, 1, (n1, m)), rng.uniform(-1, 1, (n2, m))
    g[: min(3, n1, n2)] = f[: min(3, n1, n2)]                 # exact duplicates across the operands
    d2 = cdist(f, g, metric="sqeuclidean")
    rq = sklearn_outer_kernel_matrix("rationalquadratic", f, g)
    assert np.allclose(rq, 1.0 / (1.0 + d2 / 2.0), rtol=1e-15, atol=0)
    assert np.all(rq[: min(3, n1, n2), : min(3, n1, n2)].diagonal() == 1.0)
    dot = f @ g.T
    assert np.allclose(sklearn_outer_kernel_matrix("dotproduct", f, g), 1.0 + dot, rtol=0, atol=1e-14 * (1 + m))
    assert np.allclose(sklearn_outer_kernel_matrix("pairwisekernel", f, g), dot, rtol=0, atol=1e-14 * m)
    nrm2 = np.einsum("ij,ij->i", f, f)
    assert np.array_equal(SKLEARN_OUTER["rationalquadratic"]({}).diag(f), np.ones(n1))
    assert np.allclose(SKLEARN_OUTER["dotproduct"]({}).diag(f), 1.0 + nrm2, rtol=1e-15, atol=0)
    assert np.allclose(SKLEARN_OUTER["pairwisekernel"]({}).diag(f), nrm2, rtol=1e-14, atol=0)
    # the symmetric call: RationalQuadratic fills its diagonal with exactly 1
    assert np.all(np.diagonal(sklearn_outer_kernel_matrix("rationalquadratic", f, None)) == 1.0)


def test_hyper_parameters_follow_scikit_learn():
    rng = np.random.default_rng(5)
    f, g = rng.uniform(-1, 1, (30, 12)), rng.uniform(-1, 1, (20, 12))
    d2 = cdist(f, g, metric="sqeuclidean")
    rq = sklearn_outer_kernel_matrix("rationalquadratic", f, g, length_scale=0.7, alpha=2.5)
    assert np.allclose(rq, (1.0 + d2 / (2 * 2.5 * 0.49)) ** -2.5, rtol=1e-14, atol=0)
    assert np.allclose(sklearn_outer_kernel_matrix("dotproduct", f, g, sigma_0=0.3), 0.09 + f @ g.T, rtol=0, atol=1e-14)
    # PairwiseKernel's gamma is dropped for the linear metric (filter_params=True)
    assert np.array_equal(sklearn_outer_kernel_matrix("pairwisekernel", f, g, gamma=7.0),
                          sklearn_outer_kernel_matrix("pairwisekernel", f, g))


def test_other_names_go_to_the_oracle():
    rng = np.random.default_rng(6)
    f, g = rng.uniform(-1, 1, (9, 6)), rng.uniform(-1, 1, (7, 6))
    for name in qkernels.OUTER_KERNELS:
        assert np.array_equal(sklearn_outer_kernel_matrix(name, f, g), qkernels.outer_kernel_matrix(name, f, g))
    assert math.isclose(sklearn_outer_kernel_matrix("gaussian", f[:1], f[:1])[0, 0], 1.0)


def test_quantum_kernel_oracle_with_the_scikit_learn_outer_kernels(monkeypatch):
    monkeypatch.setattr(qkernels, "outer_kernel_matrix", sklearn_outer_kernel_matrix)
    qk = qkernels.create_quantum_kernel(3, 2, 1, "yz_cx", "projected", "XYZ", "dotproduct")
    x = np.random.default_rng(1).uniform(-2, 2, (11, 2))
    qk.assign_parameters(np.linspace(0.1, 1.0, qk.encoding_circuit.num_parameters))
    K = qk.evaluate(x, x)
    fx = qk.encoding_circuit.features(x, qk.parameters)
    assert np.array_equal(K, sk.DotProduct()(fx, fx))
    assert np.all(np.diagonal(K) > 1.0)                      # sigma_0^2 + |f|^2: the diagonal is not 1


def test_outer_hyp_maps_the_new_names():
    from dqgp_b200 import _lib, kernels
    assert kernels.outer_hyp("rationalquadratic") == [1.0, 1.0]
    assert kernels.outer_hyp("rationalquadratic", {"length_scale": 0.7, "alpha": 2.5}) == [0.7, 2.5]
    assert kernels.outer_hyp("dotproduct") == [1.0]
    assert kernels.outer_hyp("dotproduct", {"sigma_0": 0.5}) == [0.5]
    assert kernels.outer_hyp("pairwisekernel") == [0.0]
    assert kernels.outer_hyp("pairwisekernel", {"gamma": 3.0, "metric": "linear"}) == [0.0]
    assert _lib.OUTER_KERNELS["rationalquadratic"] == 3
    assert _lib.OUTER_KERNELS["dotproduct"] == _lib.OUTER_KERNELS["pairwisekernel"] == 4


@pytest.mark.parametrize("metric", ["rbf", "polynomial", "cosine"])
def test_outer_hyp_rejects_non_linear_pairwise_metrics(metric):
    from dqgp_b200 import kernels
    with pytest.raises(ValueError, match="linear"):
        kernels.outer_hyp("pairwisekernel", {"metric": metric})


@pytest.mark.parametrize("name", ["whitekernel", "constantkernel", "RationalQuadratic", ""])
def test_outer_hyp_rejects_unknown_names(name):
    from dqgp_b200 import kernels
    with pytest.raises(ValueError, match="outside the hot path"):
        kernels.outer_hyp(name)
    with pytest.raises(ValueError, match="outside the hot path"):
        sklearn_outer_kernel_matrix(name, np.zeros((2, 3)), np.zeros((2, 3)))
