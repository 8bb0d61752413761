"""GPU parity, kernel level: every C-ABI compute entry point against the oracle on seeded inputs.
Tolerances: 1e-10 relative on K entries (BASELINE.json north_star), 1e-12 on features/states."""
import ctypes as C

import numpy as np
import pytest

from conftest import AGENT_CASES, load_golden

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


CIRCUITS = [("chebyshev", 3, 2, 1), ("chebyshev", 4, 2, 3), ("hubregtsen", 5, 2, 2), ("hubregtsen", 3, 5, 1),
            ("yz_cx", 8, 4, 3), ("yz_cx", 2, 1, 2), ("yz_cx", 1, 1, 1), ("kyriienko", 10, 6, 2), ("kyriienko", 6, 3, 2),
            ("hubregtsen", 7, 3, 1), ("chebyshev", 9, 4, 1), ("yz_cx", 11, 5, 1)]


@pytest.mark.parametrize("enc,q,dd,layers", CIRCUITS)
def test_features_and_states_match_oracle(d, enc, q, dd, layers):
    from oracle import circuits, statevector
    rng = np.random.default_rng(q * 100 + dd)
    n, S = 37, 5
    lo, hi = (-0.99, 0.99) if enc in ("chebyshev", "kyriienko") else (-2, 2)
    x = rng.uniform(lo, hi, (n, dd))
    P = circuits.num_parameters(enc, q, layers)
    pm = rng.uniform(0, np.pi, (S, max(P, 1)))[:, :P]
    ec = d.EncodingCircuit(enc, q, dd, layers)
    assert ec.num_parameters == P
    dx, dpm = d.kernels.dev_f64(x), d.kernels.dev_f64(pm)
    F = ec.features(dx, dpm).cpu().numpy()
    Psi = ec.states(dx, dpm).cpu().numpy()
    gates = circuits.build_circuit(enc, q, dd, layers)
    for s in range(S):
        ref = statevector.simulate(gates, q, x, pm[s])
        got = Psi[s, :, :, 0] + 1j * Psi[s, :, :, 1]
        assert np.abs(got - ref).max() < 1e-12
        assert np.abs(F[s] - statevector.pauli_features(ref, q)).max() < 1e-12


@pytest.mark.parametrize("enc,q,dd,layers", [("chebyshev", 3, 2, 1), ("chebyshev", 4, 2, 3), ("hubregtsen", 5, 2, 2), ("yz_cx", 8, 4, 3),
                                            ("yz_cx", 1, 1, 2), ("kyriienko", 10, 6, 2), ("hubregtsen", 9, 3, 1), ("yz_cx", 6, 3, 2),
                                            ("yz_cx", 12, 4, 1), ("kyriienko", 12, 6, 4),
                                            # every qubit count of the CX-free lc2 kernel (team = 1 .. 32 lanes, then a CTA)
                                            ("yz_cx", 3, 2, 2), ("kyriienko", 4, 3, 2), ("yz_cx", 5, 2, 3), ("kyriienko", 7, 4, 2),
                                            ("yz_cx", 9, 3, 2), ("kyriienko", 11, 5, 1)])
def test_shared_prefix_simulation_matches_per_set_kernels(d, enc, q, dd, layers, monkeypatch):
    """dqgp_features_shifted / dqgp_states_shifted over the 2P+1 central-difference sets against the per-set kernels:
    the two-fork prefix-sharing kernel bit for bit; the linear-combination kernel (one fork per rotation parameter, both
    signs from <psi|O|psi>, <phi|O|phi>, Re<psi|O|phi>) to rounding, including circuits whose parameters sit on CRZ gates
    (those keep two forks) and parameter sets whose +h / -h shifts wrap differently."""
    from oracle import agent_step, circuits
    rng = np.random.default_rng(7 * q + dd)
    n = 45 if q < 12 else 5
    lo, hi = (-0.99, 0.99) if enc in ("chebyshev", "kyriienko") else (-2, 2)
    x = rng.uniform(lo, hi, (n, dd))
    P = circuits.num_parameters(enc, q, layers)
    pm = agent_step.shifted_parameter_sets(np.round(rng.uniform(-0.5, 3.5, P), 4), np.pi / 8)
    ec = d.EncodingCircuit(enc, q, dd, layers)
    dx, dpm = d.kernels.dev_f64(x), d.kernels.dev_f64(pm)
    lib = d.load()
    F_ref, S_ref = ec.features(dx, dpm), ec.states(dx, dpm)
    monkeypatch.setenv("DQGP_SV_FORCE_SHARED", "1")      # n = 45 is below the size where the sharing kernels are dispatched
    for no_lc in (True, False):
        if no_lc:
            monkeypatch.setenv("DQGP_SV_NO_LC", "1")
        else:
            monkeypatch.delenv("DQGP_SV_NO_LC")
        F = torch.full_like(F_ref, float("nan"))
        S = torch.full_like(S_ref, float("nan"))
        assert lib.dqgp_features_shifted(ec.handle, dx.data_ptr(), n, dpm.data_ptr(), P, F.data_ptr(), _sp()) == 0, lib.dqgp_last_error()
        assert lib.dqgp_states_shifted(ec.handle, dx.data_ptr(), n, dpm.data_ptr(), P, S.data_ptr(), _sp()) == 0, lib.dqgp_last_error()
        torch.cuda.synchronize()
        if no_lc:
            assert torch.equal(F, F_ref)
            assert torch.equal(S, S_ref)
        else:
            assert (F - F_ref).abs().max().item() < 2e-14
            assert (S - S_ref).abs().max().item() < 2e-14
            assert torch.equal(S[0], S_ref[0])                       # the base set is simulated directly
            # ... and so are its features; the CX-free lc2 kernel (yz_cx, kyriienko: every q) sums them through the final index map
            # in another order
            assert (F[0] - F_ref[0]).abs().max().item() < 5e-15


def test_features_empty_and_single(d):
    ec = d.EncodingCircuit("yz_cx", 3, 2, 1)
    dx = d.kernels.dev_f64(np.zeros((0, 2)))
    dpm = d.kernels.dev_f64(np.zeros((1, ec.num_parameters)))
    assert ec.features(dx, dpm).shape == (1, 0, 9)
    one = ec.features(d.kernels.dev_f64(np.zeros((1, 2))), dpm).cpu().numpy()
    assert np.allclose(one[0, 0], [0, 0, 0, 0, 0, 0, 1, 1, 1])        # |000>: <Z>=1, <X>=<Y>=0


@pytest.mark.parametrize("outer", ["gaussian", "matern", "expsinesquared"])
def test_gram_projected_matches_sklearn_golden(d, outer):
    g = load_golden("outer_kernels.npz")
    F, G = g["F"], g["G"]
    lib = d.load()
    dF, dG = d.kernels.dev_f64(F), d.kernels.dev_f64(G)
    K = torch.empty((F.shape[0], G.shape[0]), dtype=torch.float64, device="cuda")
    from dqgp_b200 import _lib
    hyp = _lib.hyp_array(d.kernels.outer_hyp(outer))
    rc = lib.dqgp_gram_projected(_lib.OUTER_KERNELS[outer], hyp, dF.data_ptr(), F.shape[0], dG.data_ptr(), G.shape[0],
                                 F.shape[1], K.data_ptr(), G.shape[0], 0, _sp())
    assert rc == 0
    K = K.cpu().numpy()
    ref = g[outer]
    assert np.max(np.abs(K - ref) / np.abs(ref)) < 1e-10
    assert np.all(K[:3, -3:].diagonal() == 1.0)          # exact duplicates -> exactly outer(0) = 1


@pytest.mark.parametrize("case", AGENT_CASES)
def test_kernel_evaluate_matches_reference_K(d, case):
    """q_kernel.evaluate(X, X) through the Python mirror == the K the real reference agent computed."""
    g = load_golden(f"agent_step_{case}.npz")
    qk = d.create_quantum_kernel(int(g["q"]), int(g["d"]), int(g["layers"]), True, str(g["encoding"]), str(g["kernel_type"]),
                                 "XYZ", "gaussian")   # training Grams are Gaussian in the reference (Q1)
    qk.assign_parameters(np.mod(g["z"], np.pi))
    K = qk.evaluate(g["X"], g["X"])
    ref = g["K"]
    assert np.max(np.abs(K - ref) / np.maximum(np.abs(ref), 1e-300)) < 1e-10
    assert np.allclose(K, K.T, rtol=0, atol=1e-14)
    Kt = qk.evaluate(g["X_test"], g["X"])
    if str(g["outer_kernel"]) == "gaussian" or str(g["kernel_type"]) == "fidelity":
        assert np.max(np.abs(Kt - g["K_test_train"])) < 1e-12


def test_gram_rectangular_ragged_shapes(d):
    from oracle import qkernels
    rng = np.random.default_rng(0)
    for n1, n2 in [(1, 1), (63, 65), (64, 64), (129, 7), (5, 200)]:
        F, G = rng.uniform(-1, 1, (n1, 9)), rng.uniform(-1, 1, (n2, 9))
        ref = qkernels.outer_kernel_matrix("matern", F, G)
        from dqgp_b200 import _lib
        K = torch.full((n1, n2 + 3), -7.0, dtype=torch.float64, device="cuda")     # ld > n2, odd ld
        dF, dG = d.kernels.dev_f64(F), d.kernels.dev_f64(G)
        rc = d.load().dqgp_gram_projected(1, _lib.hyp_array([1.0]), dF.data_ptr(), n1, dG.data_ptr(), n2, 9, K.data_ptr(),
                                          n2 + 3, 0, _sp())
        assert rc == 0
        K = K.cpu().numpy()
        assert np.max(np.abs(K[:, :n2] - ref)) < 1e-13
        assert np.all(K[:, n2:] == -7.0)                  # nothing written past the logical width


@pytest.mark.parametrize("akc,bkc", [(1, 1), (1, 0), (0, 0), (0, 1)])
def test_dgemm_all_operand_layouts(d, akc, bkc):
    rng = np.random.default_rng(akc * 2 + bkc)
    M, N, K = 256, 384, 208
    A = rng.standard_normal((M, K)); B = rng.standard_normal((K, N)); Cm = rng.standard_normal((M, N))
    dA = d.kernels.dev_f64(A if akc else A.T.copy())
    dB = d.kernels.dev_f64(B.T.copy() if bkc else B)
    dC = d.kernels.dev_f64(Cm)
    rc = d.load().dqgp_dgemm(akc, bkc, M, N, K, -0.5, dA.data_ptr(), dA.shape[1], dB.data_ptr(), dB.shape[1], 2.0,
                             dC.data_ptr(), N, _sp())
    assert rc == 0, d.load().dqgp_last_error()
    ref = -0.5 * A @ B + 2.0 * Cm
    assert np.max(np.abs(dC.cpu().numpy() - ref)) < 1e-11


def test_dgemm_rejects_bad_shapes(d):
    t = torch.zeros(16, dtype=torch.float64, device="cuda")
    lib = d.load()
    assert lib.dqgp_dgemm(1, 1, 100, 128, 16, 1.0, t.data_ptr(), 16, t.data_ptr(), 16, 0.0, t.data_ptr(), 128, _sp()) < 0
    assert b"multiples" in lib.dqgp_last_error()


@pytest.mark.parametrize("dim,offset,message", [(3, 0, b"2^q"), (24, 0, b"2^q"), (8, 1, b"16-byte aligned")])
def test_fidelity_entry_points_reject_unsupported_states(d, dim, offset, message):
    """dqgp_gram_fidelity / dqgp_grad_fidelity take 2^q amplitudes (q >= 1) per state and 16-byte aligned state arrays: the DMMA
    kernel splits every state into chunks of 4k doubles and copies them with the TMA engine.  Anything else is refused before a
    launch, with a message."""
    n, P = 5, 1
    lib = d.load()
    buf = torch.zeros((2 * P + 1) * n * 2 * dim + 1, dtype=torch.float64, device="cuda")
    psi = buf[offset:offset + (2 * P + 1) * n * 2 * dim]
    assert psi.data_ptr() % 16 == 8 * offset
    K = torch.zeros((n, n), dtype=torch.float64, device="cuda")
    ainv = torch.eye(n, dtype=torch.float64, device="cuda")
    alpha = torch.zeros(n, dtype=torch.float64, device="cuda")
    grad = torch.zeros(P, dtype=torch.float64, device="cuda")
    work = torch.zeros(max(1, lib.dqgp_grad_workspace_bytes(n, P) // 8), dtype=torch.float64, device="cuda")
    assert lib.dqgp_gram_fidelity(psi.data_ptr(), n, psi.data_ptr(), n, dim, K.data_ptr(), n, 1, _sp()) < 0
    assert message in lib.dqgp_last_error()
    assert lib.dqgp_grad_fidelity(ainv.data_ptr(), n, alpha.data_ptr(), psi.data_ptr(), n, dim, P, 0.1, grad.data_ptr(),
                                  work.data_ptr(), _sp()) < 0
    assert message in lib.dqgp_last_error()
    torch.cuda.synchronize()


@pytest.mark.parametrize("n", [1, 5, 127, 128, 129, 300, 640, 1100])
def test_potrf_solve_inv_matches_lapack(d, n):
    rng = np.random.default_rng(n)
    F = rng.uniform(-1, 1, (n, 6))
    from oracle import qkernels
    A = qkernels.outer_kernel_matrix("gaussian", F, F) + 0.01 * np.eye(n)
    y = rng.standard_normal(n)
    s = d.engine.Solver(n)
    s.matrix().copy_(torch.from_numpy(A).cuda())
    f64 = dict(dtype=torch.float64, device="cuda")
    alpha, logdet, info = torch.empty(n, **f64), torch.zeros(1, **f64), torch.zeros(1, dtype=torch.int32, device="cuda")
    dy = d.kernels.dev_f64(y)
    rc = d.load().dqgp_potrf_solve_inv(s.handle, dy.data_ptr(), alpha.data_ptr(), logdet.data_ptr(), info.data_ptr(), 2, _sp())
    assert rc == 0 and int(info.item()) == 0
    L = np.linalg.cholesky(A)
    ref_alpha = np.linalg.solve(L.T, np.linalg.solve(L, y))
    ref_inv = np.linalg.solve(L.T, np.linalg.solve(L, np.eye(n)))
    sign, ref_logdet = np.linalg.slogdet(A)
    assert abs(logdet.item() - ref_logdet) < 1e-9 * max(1.0, abs(ref_logdet))
    scale = np.abs(ref_inv).max()
    assert np.max(np.abs(s.inverse().cpu().numpy() - ref_inv)) < 1e-9 * scale
    assert np.max(np.abs(alpha.cpu().numpy() - ref_alpha)) < 1e-9 * np.abs(ref_alpha).max()
    assert np.max(np.abs(np.tril(s.matrix().cpu().numpy()) - L)) < 1e-11


def test_potrf_reports_non_spd(d):
    n = 200
    A = np.eye(n); A[150, 150] = -1.0
    s = d.engine.Solver(n)
    s.matrix().copy_(torch.from_numpy(A).cuda())
    f64 = dict(dtype=torch.float64, device="cuda")
    alpha, logdet, info = torch.empty(n, **f64), torch.zeros(1, **f64), torch.zeros(1, dtype=torch.int32, device="cuda")
    dy = torch.zeros(n, **f64)
    d.load().dqgp_potrf_solve_inv(s.handle, dy.data_ptr(), alpha.data_ptr(), logdet.data_ptr(), info.data_ptr(), 0, _sp())
    assert int(info.item()) == 151


@pytest.mark.parametrize("case", AGENT_CASES)
def test_fused_gradient_matches_oracle(d, case):
    """dqgp_grad_* on the oracle's A^-1 and alpha == 1/2 sum(B * dK_i^T) with materialised dK (agent_riemannian.py:431-436)."""
    from oracle import agent_step
    g = load_golden(f"agent_step_{case}.npz")
    cfg = agent_step.KernelConfig(str(g["encoding"]), str(g["kernel_type"]), int(g["q"]), int(g["layers"]), str(g["outer_kernel"]))
    X, Y, z = g["X"], g["Y"], np.mod(g["z"], np.pi)
    K, dK = agent_step.kernel_and_derivatives(cfg, X, z, float(g["h"]))
    grad_ref, comp, _, alpha, cinv = agent_step.gp_terms(K, dK, Y, 0.1, want_cond=False)
    eng = d.AgentEngine(X, Y, encoding_type=cfg.encoding_type, kernel_type=cfg.kernel_type, num_qubits=cfg.num_qubits,
                        num_layers=cfg.num_layers, noise_std=0.1, rho=100.0, L=100.0, outer_kernel=cfg.outer_kernel)
    eng.simulate(d.kernels.dev_f64(g["z"]))
    eng.gram(); eng.factor(); eng.gradient()
    torch.cuda.synchronize()
    assert np.max(np.abs(eng.d_alpha.cpu().numpy() - alpha)) < 1e-8 * np.abs(alpha).max()
    got = eng.d_grad.cpu().numpy()
    assert np.max(np.abs(got - grad_ref)) < 1e-8 * max(1.0, np.abs(grad_ref).max())
    nll = eng.d_nll.cpu().numpy()
    assert abs(nll[3] - float(g["nll"])) < 1e-8 * max(1.0, abs(float(g["nll"])))
    assert abs(nll[0] - float(g["log_det_term"])) < 1e-8 * max(1.0, abs(float(g["log_det_term"])))
    assert abs(nll[1] - float(g["quadratic_term"])) < 1e-8 * max(1.0, abs(float(g["quadratic_term"])))
    assert nll[2] == pytest.approx(float(g["constant_term"]), rel=1e-15)


def test_admm_kernels_match_reference_golden(d):
    g = load_golden("torus.npz")
    lib = d.load()
    for c in range(4):
        theta, psi, grad, rho = g[f"c{c}_theta"], g[f"c{c}_psi"], g[f"c{c}_grad"], float(g[f"c{c}_rho"])
        A, P = theta.shape
        dz = torch.empty(P, dtype=torch.float64, device="cuda")
        dth, dps = d.kernels.dev_f64(theta), d.kernels.dev_f64(psi)
        assert lib.dqgp_admm_consensus(dth.data_ptr(), dps.data_ptr(), A, P, rho, np.pi, dz.data_ptr(), _sp()) == 0
        z_ref = np.round(g[f"c{c}_z"], 4)
        assert np.max(np.abs(dz.cpu().numpy() - z_ref)) < 1e-12          # same 1e-4 grid point
        th, ps = torch.empty(P, dtype=torch.float64, device="cuda"), torch.empty(P, dtype=torch.float64, device="cuda")
        zw = np.mod(z_ref, np.pi)
        dzw, dgr, dp0 = d.kernels.dev_f64(zw), d.kernels.dev_f64(grad), d.kernels.dev_f64(psi[0])
        assert lib.dqgp_admm_local(dzw.data_ptr(), dgr.data_ptr(), dp0.data_ptr(), P, rho, 100.0, np.pi, th.data_ptr(),
                                   ps.data_ptr(), _sp()) == 0
        assert np.array_equal(th.cpu().numpy(), np.round(g[f"c{c}_theta_new"], 4))      # bit-exact
        assert np.array_equal(ps.cpu().numpy(), np.round(g[f"c{c}_psi_new"], 4))


def test_shift_parameter_sets_bit_exact(d):
    from oracle import agent_step
    rng = np.random.default_rng(4)
    z = np.round(rng.uniform(-1, 4, 17), 4)
    ref = agent_step.shifted_parameter_sets(z, np.pi / 8)
    out = torch.empty(ref.shape, dtype=torch.float64, device="cuda")
    dz = d.kernels.dev_f64(z)
    assert d.load().dqgp_shift_parameter_sets(dz.data_ptr(), 17, np.pi / 8, np.pi, out.data_ptr(), _sp()) == 0
    assert np.array_equal(out.cpu().numpy(), ref)


@pytest.mark.parametrize("n,ob", [(100, 4), (640, 1), (1500, 2), (2100, 4), (4500, -1)])
def test_lean_solver_matches_full_solver(d, n, ob):
    """Lean solver (one square, rotating panel buffers, substitution solves) == full solver: same factor bit for bit,
    alpha / logdet to rounding, and the in-place quadratic form == the L^-1-based one."""
    from dqgp_b200.engine import Solver
    lib = d.load()
    rng = np.random.default_rng(n)
    B = rng.standard_normal((n, 40))
    A = B @ B.T / 40 + np.eye(n)
    y = rng.standard_normal(n)
    rhs = rng.standard_normal((70, n))
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = {}
    for lean in (False, True):
        s = Solver(n, ob, lean=lean)
        assert lib.dqgp_solver_is_lean(s.handle) == int(lean)
        s.matrix().copy_(torch.from_numpy(A).cuda())
        alpha = torch.empty(n, dtype=torch.float64, device="cuda")
        logdet = torch.zeros(1, dtype=torch.float64, device="cuda")
        info = torch.zeros(1, dtype=torch.int32, device="cuda")
        assert lib.dqgp_potrf_solve_inv(s.handle, torch.from_numpy(y).cuda().data_ptr(), alpha.data_ptr(), logdet.data_ptr(),
                                        info.data_ptr(), 0, st) == 0
        torch.cuda.synchronize()
        assert info.item() == 0
        L = np.tril(s.matrix().cpu().numpy())
        nbp, ld = 128, s.ld
        Bp = torch.zeros((nbp, ld), dtype=torch.float64, device="cuda")
        Bp[:70, :n] = torch.from_numpy(rhs).cuda()
        q = torch.empty(nbp, dtype=torch.float64, device="cuda")
        assert lib.dqgp_solver_quadform_rows_inplace(s.handle, Bp.data_ptr(), nbp, ld, q.data_ptr(), st) == 0
        torch.cuda.synchronize()
        out[lean] = (L, alpha.cpu().numpy(), logdet.item(), q.cpu().numpy()[:70], Bp.cpu().numpy()[:70, :n])
        if not lean:
            q2 = torch.empty(70, dtype=torch.float64, device="cuda")
            assert lib.dqgp_solver_quadform_rows(s.handle, torch.from_numpy(rhs).cuda().data_ptr(), 70, n, q2.data_ptr(), st) == 0
            assert np.max(np.abs(q2.cpu().numpy() - out[lean][3]) / out[lean][3]) < 1e-11
        else:
            # a lean solver refuses what it cannot do
            assert lib.dqgp_potrf_solve_inv(s.handle, torch.from_numpy(y).cuda().data_ptr(), alpha.data_ptr(), logdet.data_ptr(),
                                            info.data_ptr(), 1, st) < 0
            assert lib.dqgp_solver_inverse(s.handle) is None
    Lf, af, ldf, qf, vf = out[False]
    Ll, al, ldl, ql, vl = out[True]
    assert np.array_equal(Lf, Ll)
    assert ldf == ldl
    Lref = np.linalg.cholesky(A)
    assert np.max(np.abs(Ll - Lref)) < 1e-11
    aref = np.linalg.solve(A, y)
    assert np.max(np.abs(al - aref)) / np.max(np.abs(aref)) < 1e-11
    assert np.max(np.abs(af - al)) / np.max(np.abs(aref)) < 1e-12
    import scipy.linalg as sl
    vref = sl.solve_triangular(Lref, rhs.T, lower=True).T
    assert np.max(np.abs(vl - vref)) < 1e-10
    assert np.max(np.abs(ql - (vref ** 2).sum(axis=1)) / ql) < 1e-11
    assert np.array_equal(vf, vl)


@pytest.mark.parametrize("enc,q,dd,layers", [("yz_cx", 4, 3, 2), ("kyriienko", 3, 2, 2), ("yz_cx", 9, 3, 1), ("yz_cx", 8, 4, 3),
                                            ("chebyshev", 4, 2, 3), ("hubregtsen", 5, 2, 2), ("chebyshev", 3, 2, 1), ("hubregtsen", 9, 3, 1)])
def test_feature_jacobian_matches_finite_differences(d, enc, q, dd, layers):
    """dqgp_features_jacobian (exact derivative of every Pauli feature with respect to every circuit parameter, from the
    cross term Re<psi|O|phi> of the linear-combination simulator) against central differences of dqgp_features."""
    rng = np.random.default_rng(3 * q + dd)
    n = 37
    lo, hi = (-0.99, 0.99) if enc in ("kyriienko", "chebyshev") else (-2, 2)
    x = rng.uniform(lo, hi, (n, dd))
    ec = d.EncodingCircuit(enc, q, dd, layers)
    P = ec.num_parameters
    p = rng.uniform(0.1, 3.0, P)
    lib = d.load()
    dx, dp = d.kernels.dev_f64(x), d.kernels.dev_f64(p)
    F = torch.full((n, 3 * q), float("nan"), dtype=torch.float64, device="cuda")
    J = torch.full((P, n, 3 * q), float("nan"), dtype=torch.float64, device="cuda")
    assert lib.dqgp_features_jacobian(ec.handle, dx.data_ptr(), n, dp.data_ptr(), F.data_ptr(), J.data_ptr(), _sp()) == 0, lib.dqgp_last_error()
    h = 1e-6
    sets = np.tile(p, (2 * P + 1, 1))
    for i in range(P):
        sets[1 + 2 * i, i] += h
        sets[2 + 2 * i, i] -= h
    Fs = ec.features(dx, d.kernels.dev_f64(sets))
    torch.cuda.synchronize()
    assert torch.equal(F, Fs[0])
    fd = (Fs[1::2] - Fs[2::2]) / (2 * h)
    assert (J - fd).abs().max().item() < 5e-9
    assert J.abs().max().item() > 1e-3


@pytest.mark.parametrize("ob", [1, 2, 4, -1])
def test_lookahead_cholesky_is_deterministic_at_full_size(d, ob):
    """The three-stream look-ahead schedule orders every writer of a block with events: the factor of an 8192 x 8192 matrix
    (config 4's shard size, 64 leaves) must be bit-identical run to run, for every outer-panel width, and a solve of it must
    reproduce the right-hand side."""
    from dqgp_b200.engine import Solver
    lib = d.load()
    n = 8192
    g = torch.Generator(device="cuda").manual_seed(3)
    B = torch.randn((n, 96), dtype=torch.float64, device="cuda", generator=g)
    A = B @ B.T / 96 + 0.05 * torch.eye(n, dtype=torch.float64, device="cuda")
    y = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
    s = Solver(n, ob)
    alpha = torch.empty(n, dtype=torch.float64, device="cuda")
    logdet = torch.zeros(1, dtype=torch.float64, device="cuda")
    info = torch.zeros(1, dtype=torch.int32, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    outs = []
    for rep in range(3):
        s.matrix().copy_(A)
        assert lib.dqgp_potrf_solve_inv(s.handle, y.data_ptr(), alpha.data_ptr(), logdet.data_ptr(), info.data_ptr(), 1, st) == 0
        torch.cuda.synchronize()
        assert info.item() == 0
        outs.append((torch.tril(s.matrix()).clone(), torch.tril(s.inverse()).clone(), alpha.clone(), logdet.item()))
    for o in outs[1:]:
        assert torch.equal(o[0], outs[0][0]) and torch.equal(o[1], outs[0][1]) and torch.equal(o[2], outs[0][2]) and o[3] == outs[0][3]
    assert ((A @ outs[0][2] - y).abs().max() / y.abs().max()).item() < 1e-9


@pytest.mark.parametrize("outer", ["matern", "expsinesquared"])
@pytest.mark.parametrize("enc,q,dd,layers,n", [("kyriienko", 4, 6, 2, 150), ("chebyshev", 3, 2, 1, 97), ("yz_cx", 5, 4, 2, 200),
                                                ("hubregtsen", 3, 4, 2, 64)])
def test_fused_gradient_honoured_outer_kernels_match_oracle(d, outer, enc, q, dd, layers, n):
    """The Matern (OUTER = 1) and ExpSineSquared (OUTER = 2) instantiations of the fused gradient, i.e. training Grams that
    HONOUR --outer-kernel (training_ignores_outer_kernel=False; the reference's Q1 default is tested above): dqgp_grad_projected
    on the ORACLE's C^-1 and alpha equals 1/2 sum(B o dK_i^T) with the oracle's materialised dK (agent_riemannian.py:431-436) to
    1e-8.  ExpSineSquared Grams are indefinite, so the oracle's C^-1 comes from the reference's LU branch (:419-425) — the kernel
    under test is the contraction, fed the same operands."""
    from oracle import agent_step
    x, y = d.synthetic_dataset(n, dd, enc, seed=n)
    cfg = agent_step.KernelConfig(enc, "projected", q, layers, outer, training_ignores_outer_kernel=False)
    eng = d.AgentEngine(x, y, encoding_type=enc, kernel_type="projected", num_qubits=q, num_layers=layers, noise_std=0.1, rho=100.0,
                        L=100.0, outer_kernel=outer, training_ignores_outer_kernel=False)
    z = np.round(np.random.RandomState(n).rand(eng.P) * np.pi, 4)
    K, dK = agent_step.kernel_and_derivatives(cfg, x, np.mod(z, np.pi), np.pi / 8)
    grad_ref, comp, _, alpha, cinv = agent_step.gp_terms(K, dK, y, 0.1, want_cond=False)
    eng.simulate(d.kernels.dev_f64(z))
    eng.gram()
    Kd = torch.tril(eng.solver.matrix()).cpu().numpy()
    ref_l = np.tril(K + 0.01 * np.eye(n))
    assert np.max(np.abs(Kd - ref_l) / np.maximum(np.abs(ref_l), 1e-300)) < 1e-10
    eng.solver.inverse().copy_(torch.from_numpy(cinv).cuda())
    eng.d_alpha.copy_(torch.from_numpy(alpha).cuda())
    eng.gradient()
    torch.cuda.synchronize()
    got = eng.d_grad.cpu().numpy()
    assert np.max(np.abs(got - grad_ref)) < 1e-8 * max(1.0, np.abs(grad_ref).max())
    if outer == "matern":          # positive definite: the whole device path (Cholesky, alpha, inverse, NLL) as well
        eng.factor(); eng.gradient()
        torch.cuda.synchronize(); eng.check_info()
        assert np.max(np.abs(eng.d_grad.cpu().numpy() - grad_ref)) < 1e-8 * max(1.0, np.abs(grad_ref).max())
        assert abs(float(eng.d_nll[3].item()) - comp["total"]) < 1e-8 * max(1.0, abs(comp["total"]))
    else:                          # indefinite: the Cholesky must report it, and the LU rung (as the oracle's gp_terms) must agree
        eng.gram(); eng.factor()
        torch.cuda.synchronize()
        assert int(eng.d_info.item()) > 0
        eng.gram(full=True); eng.factor_lu(); eng.gradient()
        torch.cuda.synchronize()
        assert np.max(np.abs(eng.d_alpha.cpu().numpy() - alpha)) < 1e-8 * np.abs(alpha).max()
        assert np.max(np.abs(eng.d_grad.cpu().numpy() - grad_ref)) < 1e-8 * max(1.0, np.abs(grad_ref).max())
        if np.isfinite(comp["total"]):
            assert abs(float(eng.d_nll[3].item()) - comp["total"]) < 1e-8 * max(1.0, abs(comp["total"]))


@pytest.mark.parametrize("enc,ktype,q,dd,layers,n,outer", [("yz_cx", "projected", 8, 4, 3, 333, "gaussian"), ("kyriienko", "projected", 10, 6, 2, 200, "matern"),
                                                          ("yz_cx", "projected", 5, 3, 2, 64, "expsinesquared"), ("hubregtsen", "fidelity", 5, 2, 2, 333, "gaussian"),
                                                          ("chebyshev", "fidelity", 2, 2, 1, 97, "gaussian")])
def test_gradient_staging_paths_agree_bit_for_bit(d, enc, ktype, q, dd, layers, n, outer):
    """The fused projected gradient stages its feature tiles through a 3-D tensor map (TMA: even m, 16-byte aligned features) or
    through per-thread cp.async (any other features): same arithmetic on the same operands, so the gradients must be identical to the
    last bit - at ragged n, where the tensor map zero-fills the rows past n and cp.async clamps them.  The fused fidelity gradient has
    one staging path (the tensor map); it is checked against the central difference assembled from the per-set Grams, whose tiles
    arrive as one bulk copy per row."""
    x, y = d.synthetic_dataset(n, dd, enc, seed=3)
    eng = d.AgentEngine(x, y, encoding_type=enc, kernel_type=ktype, num_qubits=q, num_layers=layers, noise_std=0.1, rho=100.0, L=100.0,
                        outer_kernel=outer, training_ignores_outer_kernel=False)
    z = d.kernels.dev_f64(np.round(np.random.RandomState(1).rand(eng.P) * np.pi, 4))
    eng.simulate(z); eng.gram(full=True)
    rs = np.random.RandomState(2)                       # any symmetric "inverse" and alpha will do: the contraction is what is compared
    b = rs.randn(n, n)
    ainv, alpha = b + b.T, rs.randn(n)
    eng.solver.inverse()[:n, :n].copy_(torch.from_numpy(ainv).cuda())
    eng.d_alpha.copy_(torch.from_numpy(alpha).cuda())
    eng.d_grad.zero_()
    eng.gradient()
    torch.cuda.synchronize()
    got = eng.d_grad.cpu().numpy().copy()
    assert np.all(np.isfinite(got)) and np.abs(got).max() > 0
    lib, s = d.load(), eng.solver
    if ktype == "projected":
        # the same features at an 8-byte offset: not 16-byte aligned, so the cp.async kernel
        buf = torch.empty(eng.d_feat.numel() + 1, dtype=torch.float64, device="cuda")
        feat = buf[1:].view(eng.d_feat.shape)
        feat.copy_(eng.d_feat)
        assert feat.data_ptr() % 16 == 8
        grad = torch.zeros_like(eng.d_grad)
        assert lib.dqgp_grad_projected(eng._outer_id, eng._hyp, s.inverse_ptr, s.ld, eng.d_alpha.data_ptr(), feat.data_ptr(), n, eng.m,
                                       eng.P, eng.h, grad.data_ptr(), eng.d_work.data_ptr(), _sp()) == 0, lib.dqgp_last_error()
        torch.cuda.synchronize()
        assert np.array_equal(got, grad.cpu().numpy())
    else:
        dim = 1 << q
        K = torch.empty((eng.S, n, n), dtype=torch.float64, device="cuda")
        for st in range(eng.S):
            f = eng.d_feat[st].data_ptr()
            assert lib.dqgp_gram_fidelity(f, n, f, n, dim, K[st].data_ptr(), n, 1, _sp()) == 0, lib.dqgp_last_error()
        torch.cuda.synchronize()
        K = K.cpu().numpy()
        bracket = ainv - np.outer(alpha, alpha)
        ref = np.array([0.5 * np.sum(bracket * (K[1 + 2 * i] - K[2 + 2 * i])) / (2.0 * eng.h) for i in range(eng.P)])
        assert np.max(np.abs(got - ref)) <= 1e-12 * np.abs(ref).max()


@pytest.mark.parametrize("n", [1, 5, 33, 64, 100, 257, 700])
@pytest.mark.parametrize("kind", ["indefinite", "general"])
def test_lu_solve_inv_matches_lapack(d, n, kind):
    """dqgp_lu_solve_inv (the reference's LU rung, agent_riemannian.py:419-425 / main.py:1479-1486) against LAPACK through
    SciPy / NumPy: alpha = lu_solve(lu_factor(A), y), A^-1 = lu_solve(lu, eye), slogdet."""
    from scipy.linalg import lu_factor, lu_solve
    rng = np.random.default_rng(n)
    if kind == "indefinite":
        q, _ = np.linalg.qr(rng.standard_normal((n, n)))
        lam = rng.uniform(0.5, 20.0, n) * np.where(rng.random(n) < 0.3, -1.0, 1.0)
        A = (q * lam) @ q.T
        A = 0.5 * (A + A.T)
    else:
        A = rng.standard_normal((n, n)) + 0.1 * np.eye(n)
    y = rng.standard_normal(n)
    lu = lu_factor(A)
    alpha_ref, inv_ref = lu_solve(lu, y), lu_solve(lu, np.eye(n))
    sign_ref, logabs_ref = np.linalg.slogdet(A)
    ld = n + 3                                   # a leading dimension that is not n
    f64 = dict(dtype=torch.float64, device="cuda")
    dA = torch.zeros((n, ld), **f64); dA[:, :n] = torch.from_numpy(A).cuda()
    dinv, dalpha, dsl = torch.full((n, ld), 7.0, **f64), torch.empty(n, **f64), torch.empty(2, **f64)
    lib = d.load()
    work = torch.empty(int(lib.dqgp_lu_workspace_bytes(n)) // 8 + 2, **f64)
    dy = torch.from_numpy(y).cuda()
    assert lib.dqgp_lu_solve_inv(dA.data_ptr(), ld, n, dy.data_ptr(), dalpha.data_ptr(), dinv.data_ptr(), ld, dsl.data_ptr(),
                                 work.data_ptr(), _sp()) == 0
    torch.cuda.synchronize()
    scale = np.abs(inv_ref).max()
    assert np.max(np.abs(dinv[:, :n].cpu().numpy() - inv_ref)) < 1e-9 * scale
    assert torch.all(dinv[:, n:] == 7.0)                                      # nothing written past the n columns
    assert np.max(np.abs(dalpha.cpu().numpy() - alpha_ref)) < 1e-9 * max(1.0, np.abs(alpha_ref).max())
    sl = dsl.cpu().numpy()
    assert sl[1] == sign_ref and abs(sl[0] - logabs_ref) < 1e-10 * max(1.0, abs(logabs_ref))
    # the L and U factors themselves equal LAPACK's (same pivot rule): compare the packed factor
    assert np.max(np.abs(dA[:, :n].cpu().numpy() - lu[0])) < 1e-9 * max(1.0, np.abs(lu[0]).max())


def test_dgemm_general_and_rowdot(d):
    rng = np.random.default_rng(1)
    M, N, K = 37, 91, 53
    A, B, C = rng.standard_normal((M, K)), rng.standard_normal((K, N)), rng.standard_normal((M, N))
    dA, dB, dC = (torch.from_numpy(v).cuda() for v in (A, B, C))
    lib = d.load()
    assert lib.dqgp_dgemm_general(M, N, K, -0.5, dA.data_ptr(), K, dB.data_ptr(), N, 2.0, dC.data_ptr(), N, _sp()) == 0
    assert np.max(np.abs(dC.cpu().numpy() - (2.0 * C - 0.5 * A @ B))) < 1e-12
    out = torch.empty(M, dtype=torch.float64, device="cuda")
    assert lib.dqgp_rowdot(dA.data_ptr(), K, dA.data_ptr(), K, M, K, out.data_ptr(), _sp()) == 0
    assert np.max(np.abs(out.cpu().numpy() - (A * A).sum(axis=1))) < 1e-12
