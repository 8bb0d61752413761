"""GPU tests of the analytic NLL gradient of the fidelity kernel (AgentEngine(kernel_type="fidelity", gradient="analytic")) for every
qubit count: dqgp_states_jacobian at 7 to 12 qubits against differences of dqgp_states, dqgp_grad_fidelity_analytic on both of its
paths (the per-row kernel for 2^q <= 64, the two DMMA stages above) against a torch complex128 formula, the engine against the
oracle's NLL, and the CUDA-graph replays of RiemannianAgent and AdmmEngine in this mode."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def d():
    import dqgp_b200
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")
    return dqgp_b200


def _sp():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("enc,q,dd,layers", [("hubregtsen", 7, 2, 2), ("yz_cx", 7, 3, 1), ("chebyshev", 8, 2, 1), ("kyriienko", 8, 4, 1),
                                            ("hubregtsen", 9, 3, 1), ("yz_cx", 10, 2, 1), ("chebyshev", 10, 2, 1), ("hubregtsen", 12, 2, 1),
                                            ("yz_cx", 12, 2, 1)])
def test_states_jacobian_matches_differences_of_the_states(d, enc, q, dd, layers):
    """dqgp_states_jacobian at the lane-group (q = 7, 8) and CTA (q = 9 to 12) sizes of the simulator: the states equal dqgp_states
    at the same parameters bit for bit, and d psi / dp_i equals central differences of dqgp_states (h = 1e-6)."""
    rng = np.random.default_rng(11 * q + dd)
    n = 37
    lo, hi = (-0.99, 0.99) if enc in ("kyriienko", "chebyshev") else (-2, 2)
    x = rng.uniform(lo, hi, (n, dd))
    ec = d.EncodingCircuit(enc, q, dd, layers)
    P, dim = ec.num_parameters, 1 << q
    p = rng.uniform(0.1, 3.0, P)
    lib = d.load()
    dx, dp = d.kernels.dev_f64(x), d.kernels.dev_f64(p)
    psi = torch.full((n, dim, 2), float("nan"), dtype=torch.float64, device="cuda")
    D = torch.full((P, n, dim, 2), float("nan"), dtype=torch.float64, device="cuda")
    assert lib.dqgp_states_jacobian(ec.handle, dx.data_ptr(), n, dp.data_ptr(), psi.data_ptr(), D.data_ptr(), _sp()) == 0, lib.dqgp_last_error()
    assert torch.equal(psi, ec.states(dx, dp.reshape(1, P))[0])
    h = 1e-6
    for i in range(P):
        sets = np.tile(p, (2, 1))
        sets[0, i] += h
        sets[1, i] -= h
        s = ec.states(dx, d.kernels.dev_f64(sets))
        fd = (s[0] - s[1]) / (2 * h)
        assert (D[i] - fd).abs().max().item() < 5e-9 * max(D.abs().max().item(), 1e-300), i
    torch.cuda.synchronize()
    assert D.abs().max().item() > 1e-3


def _states(rng, n, dim, P):
    psi = rng.standard_normal((n, dim)) + 1j * rng.standard_normal((n, dim))
    psi /= np.linalg.norm(psi, axis=1, keepdims=True)
    D = rng.standard_normal((P, n, dim)) + 1j * rng.standard_normal((P, n, dim))
    A = rng.standard_normal((n, n))
    return psi, D / np.sqrt(dim), A + A.T, rng.standard_normal(n)


def _reference(psi, D, Ainv, alpha):
    """S = Psi Psi^H, W = B o S, G = W Psi, grad_i = 2 Re sum conj(G) D_i in torch complex128 on the device."""
    P_ = torch.from_numpy(psi).cuda()
    D_ = torch.from_numpy(D).cuda()
    B = torch.from_numpy(Ainv - np.outer(alpha, alpha)).cuda()
    G = (B * (P_ @ P_.conj().T)) @ P_
    return (2.0 * (G.conj().unsqueeze(0) * D_).real.sum(dim=(1, 2))).cpu().numpy()


def _c2r(z):
    return np.ascontiguousarray(np.stack([z.real, z.imag], axis=-1))


def _device(d, psi, D, Ainv, alpha, psi_offset=0):
    """dqgp_grad_fidelity_analytic with ld = n + 3 (NaN in the padding columns of A^-1); returns (rc, gradient)."""
    lib = d.load()
    n, dim = psi.shape
    P = D.shape[0]
    ld = n + 3
    A = np.full((n, ld), np.nan)
    A[:, :n] = Ainv
    dA, dal, dD = (d.kernels.dev_f64(v) for v in (A, alpha, _c2r(D)))
    buf = torch.empty(n * dim * 2 + 2, dtype=torch.float64, device="cuda")
    dpsi = buf[psi_offset:psi_offset + n * dim * 2]
    dpsi.copy_(torch.from_numpy(_c2r(psi).reshape(-1)).cuda())
    work = torch.empty(lib.dqgp_grad_fidelity_analytic_workspace_bytes(n, dim) // 8 + 1, dtype=torch.float64, device="cuda")
    grad = torch.full((P,), -7.0, dtype=torch.float64, device="cuda")
    rc = lib.dqgp_grad_fidelity_analytic(dA.data_ptr(), ld, dal.data_ptr(), dpsi.data_ptr(), dD.data_ptr(), n, dim, P, grad.data_ptr(),
                                         work.data_ptr(), _sp())
    torch.cuda.synchronize()
    return rc, grad.cpu().numpy()


@pytest.mark.parametrize("dim", [1 << q for q in range(1, 13)])
def test_abi_matches_an_independent_formula(d, dim):
    """Both paths (per-row kernel up to 2^q = 64, weights + GEMM + contraction above) against torch complex128, to 1e-10 of the
    largest gradient entry, for ragged n, an exact multiple of the 128-row tile and ld > n; a second call gives the same bits."""
    rng = np.random.default_rng(dim)
    lib = d.load()
    for n in [37, 130, 300, 256]:
        psi, D, Ainv, alpha = _states(rng, n, dim, 3)
        ref = _reference(psi, D, Ainv, alpha)
        rc, got = _device(d, psi, D, Ainv, alpha)
        assert rc == 0, lib.dqgp_last_error()
        assert np.all(np.abs(got - ref) <= 1e-10 * np.abs(ref).max()), (n, got, ref)
        assert np.array_equal(got, _device(d, psi, D, Ainv, alpha)[1])


@pytest.mark.parametrize("dim", [64, 256])
def test_nan_amplitude_reaches_the_gradient(d, dim):
    rng = np.random.default_rng(5)
    psi, D, Ainv, alpha = _states(rng, 70, dim, 4)
    psi[5, 3] = complex(np.nan, 0.0)
    rc, got = _device(d, psi, D, Ainv, alpha)
    assert rc == 0 and np.all(np.isnan(got))


@pytest.mark.parametrize("dim,offset,message", [(96, 0, b"2^q"), (8192, 0, b"2^q"), (128, 1, b"16-byte aligned")])
def test_abi_rejects_unsupported_arguments(d, dim, offset, message):
    """dim must be 2^q with q <= 12, and from 2^q = 128 on the states must be 16-byte aligned (their tiles arrive by TMA)."""
    lib = d.load()
    n, P = 5, 2
    psi = torch.zeros(n * dim * 2 + 1, dtype=torch.float64, device="cuda")[offset:]
    assert psi.data_ptr() % 16 == 8 * offset
    D = torch.zeros(P * n * dim * 2, dtype=torch.float64, device="cuda")
    ainv = torch.eye(n, dtype=torch.float64, device="cuda")
    alpha = torch.zeros(n, dtype=torch.float64, device="cuda")
    grad = torch.zeros(P, dtype=torch.float64, device="cuda")
    work = torch.zeros(16, dtype=torch.float64, device="cuda")
    assert lib.dqgp_grad_fidelity_analytic(ainv.data_ptr(), n, alpha.data_ptr(), psi.data_ptr(), D.data_ptr(), n, dim, P, grad.data_ptr(),
                                           work.data_ptr(), _sp()) < 0
    assert message in lib.dqgp_last_error()
    torch.cuda.synchronize()


def test_small_state_workspace_is_unchanged(d):
    """Up to 2^q = 64 the per-row kernel keeps its workspace: 16 segment partials plus the sum, complex, per sample and amplitude."""
    lib = d.load()
    for n in [1, 37, 300, 8192]:
        for dim in [2, 4, 8, 16, 32, 64]:
            assert lib.dqgp_grad_fidelity_analytic_workspace_bytes(n, dim) == 8 * 2 * 17 * n * dim
        npad = (n + 127) // 128 * 128
        for dim in [128, 4096]:
            assert lib.dqgp_grad_fidelity_analytic_workspace_bytes(n, dim) == 8 * (16 + 2 * npad * npad + 6 * npad * dim)


def _oracle_nll(x, y, q, dd, layers, enc, p):
    from oracle import qkernels
    qk = qkernels.create_quantum_kernel(q, dd, layers, enc, "fidelity", "XYZ", "gaussian")
    qk.assign_parameters(p)
    a = qk.evaluate(x, x) + 0.01 * np.eye(len(y))
    L = np.linalg.cholesky(a)
    return np.log(np.diag(L)).sum() + 0.5 * y @ np.linalg.solve(a, y) + 0.5 * len(y) * np.log(2 * np.pi)


@pytest.mark.parametrize("enc,q,dd,layers,n", [("hubregtsen", 7, 2, 2, 120), ("chebyshev", 7, 2, 1, 100), ("yz_cx", 8, 2, 1, 160),
                                                ("hubregtsen", 8, 2, 2, 140), ("chebyshev", 10, 2, 1, 40)])
def test_engine_gradient_is_the_derivative_of_the_oracle_nll(d, enc, q, dd, layers, n):
    """AgentEngine(kernel_type="fidelity", gradient="analytic") from 7 qubits on (hubregtsen with two layers: with one, its trainable
    gates follow the encoding and the fidelity kernel does not depend on them): the NLL equals the oracle's, the gradient equals
    central differences of the oracle's NumPy/LAPACK NLL, the central-difference mode gives a visibly different number, and the
    LU rung (step_fallback) gives the Cholesky step's gradient."""
    x, y = d.synthetic_dataset(n, dd, enc)
    P = d.EncodingCircuit(enc, q, dd, layers).num_parameters
    z = np.round(np.random.RandomState(5).uniform(0.2, 2.9, P), 4)
    dz, dpsi = d.kernels.dev_f64(z), d.kernels.dev_f64(np.zeros(P))
    theta, psi_out = torch.empty_like(dz), torch.empty_like(dz)
    grads = {}
    for mode in ("analytic", "central_difference"):
        eng = d.AgentEngine(x, y, encoding_type=enc, kernel_type="fidelity", num_qubits=q, num_layers=layers, noise_std=0.1, rho=100.0,
                            L=100.0, gradient=mode)
        eng.step(dz, dpsi, theta, psi_out)
        torch.cuda.synchronize(); eng.check_info()
        grads[mode] = eng.d_grad.cpu().numpy().copy()
        if mode == "analytic":
            nll_gpu = float(eng.d_nll[3].item())
            eng.step_fallback(dz, dpsi, theta, psi_out)
            torch.cuda.synchronize()
            assert eng.used_lu_fallback
            g_lu = eng.d_grad.cpu().numpy()
            assert np.max(np.abs(g_lu - grads["analytic"])) <= 1e-10 * np.max(np.abs(grads["analytic"]))
    assert np.abs(grads["analytic"]).max() > 1e-6
    ref_nll = _oracle_nll(x, y, q, dd, layers, enc, z)
    assert abs(ref_nll - nll_gpu) < 1e-8 * abs(nll_gpu)
    h = 1e-5
    for i in range(0, P, max(1, P // 5)):
        e = np.zeros_like(z); e[i] = h
        ref = (_oracle_nll(x, y, q, dd, layers, enc, z + e) - _oracle_nll(x, y, q, dd, layers, enc, z - e)) / (2 * h)
        assert abs(grads["analytic"][i] - ref) < 2e-5 * max(1.0, abs(ref)), (i, grads["analytic"][i], ref)
    assert np.max(np.abs(grads["analytic"] - grads["central_difference"])) > 1e-3 * np.max(np.abs(grads["analytic"]))


def test_riemannian_agent_reference_defaults_at_7_qubits(d):
    """RiemannianAgent(kernel_type="fidelity", use_parameter_shift=False), the reference's defaults, maps to the analytic gradient
    and runs at 7 qubits; its second call (a CUDA-graph replay) returns what the eager first call returned."""
    x, y = d.synthetic_dataset(130, 2, "yz_cx")
    rs = np.random.RandomState(3)
    P = d.EncodingCircuit("yz_cx", 7, 2, 2).num_parameters
    z, psi = np.round(rs.uniform(0.2, 2.9, P), 4), np.round(rs.rand(P), 4)
    ag = d.RiemannianAgent("fid7", x, y, 7, 0.1, 100.0, 100.0, kernel_type="fidelity", use_parameter_shift=False, num_layers=2)
    assert ag.gradient == "analytic"
    eager = ag.train_and_update(z, psi)
    g_eager = ag.last_gradient.copy()
    assert ag._engine()._graph is None
    replayed = ag.train_and_update(z, psi)
    assert ag._engine()._graph is not None
    for a, b in zip(eager[:3], replayed[:3]):
        assert np.array_equal(a, b)
    assert np.array_equal(g_eager, ag.last_gradient)
    assert np.all(np.isfinite(g_eager)) and np.abs(g_eager).max() > 0


@pytest.mark.parametrize("q", [5, 7])
def test_admm_engine_graph_replay_equals_eager_iterations(d, q):
    """AdmmEngine.capture()/replay() in analytic fidelity mode walks the same trajectory as eager iteration() calls, on the per-row
    path (q = 5) and on the DMMA path (q = 7)."""
    x, y = d.synthetic_dataset(3 * 140, 2, "hubregtsen")
    shards = [(x[a * 140:(a + 1) * 140], y[a * 140:(a + 1) * 140]) for a in range(3)]
    P = d.EncodingCircuit("hubregtsen", q, 2, 2).num_parameters
    rs = np.random.RandomState(q)
    theta0, psi0 = np.round(rs.rand(3, P), 4), np.round(rs.rand(3, P), 4)
    kw = dict(rho=100.0, L=100.0, encoding_type="hubregtsen", kernel_type="fidelity", num_qubits=q, num_layers=2, noise_std=0.1,
              gradient="analytic")
    eager = d.AdmmEngine(shards, theta0, psi0, **kw)
    for _ in range(3):
        eager.iteration()
    graph = d.AdmmEngine(shards, theta0, psi0, **kw)
    graph.capture()
    for _ in range(3):
        graph.replay()
    for a, b in zip(eager.state(), graph.state()):
        assert np.array_equal(a, b)
    assert all(ag.gradient_mode == "analytic" for ag in graph.agents)
    assert any(np.abs(ag.d_grad.cpu().numpy()).max() > 1e-6 for ag in graph.agents)
