"""GPU tests of the analytic NLL gradients at the shard sizes they run at: dqgp_grad_projected_analytic (every outer id),
dqgp_grad_fidelity_analytic (the per-row path at config 3's 2^q = 32 and the DMMA path at 2^q = 128 and 1024),
dqgp_grad_outer_hyperparameters and dqgp_grad_noise_std, on the inputs a real step gives them: A^-1 and alpha from the
factorisation of K + sigma^2 I (sigma = 0.1), the simulator's features or states and their Jacobian.

Sizes: n = 8192 (configs 4 and 5), 2048 (config 3), 2053 and 8192 on the DMMA path, and the ragged 1025, 4099 and 8193.  Below
n = 1025 every 16-way column segment of the per-row kernels is one shared-memory chunk; these sizes run 2 to 8 chunks per segment,
ragged last chunks and ragged last segments.

Each ABI result is compared with a reference that shares no code with the kernels (closed forms of scikit-learn's kernels,
torch float64 / complex128 on the device), to a bound derived from the sum of absolute terms T_i (see _bound_doc), and the
engine's analytic gradient is compared with Richardson-extrapolated central differences of the device's own
central-difference path and NLL."""
import ctypes as C
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

U = 2.0 ** -53
GA_SEGMENTS, GA_CHUNK, GF_CHUNK, GM_BM, GFD_SLICES = 16, 64, 16, 128, 64      # grad.cu's partition of the work
GROUP = 8                               # the references add in a tree of groups of 8 (_tree_sum)
C_W = 16                                # ulp of one outer-kernel weight for an exact argument (_bound_doc)
C_Y = 8                                 # roundings in the argument of the weight's exponent (_bound_doc)
SIGMA = 0.1

# name: (encoding, kernel type, q, layers, d, n, outer kernel of the training Gram)
SHARDS = {
    "cfg4": ("yz_cx", "projected", 8, 3, 4, 8192, "gaussian"),
    "cfg5": ("kyriienko", "projected", 10, 4, 6, 8192, "matern"),
    "cfg4-1025": ("yz_cx", "projected", 8, 3, 4, 1025, "gaussian"),
    "cfg5-4099": ("kyriienko", "projected", 10, 4, 6, 4099, "matern"),
    "cfg4-8193": ("yz_cx", "projected", 8, 3, 4, 8193, "gaussian"),
    "cfg3": ("hubregtsen", "fidelity", 5, 2, 2, 2048, None),
    "fid-q7-2053": ("hubregtsen", "fidelity", 7, 2, 2, 2053, None),
    "fid-q10-2053": ("hubregtsen", "fidelity", 10, 2, 2, 2053, None),
    "fid-q7-8192": ("hubregtsen", "fidelity", 7, 2, 2, 8192, None),
}

# (outer id name, hyper-parameters in h_hyp order): the default and one non-default set of every outer id
OUTER_CASES = [("gaussian", [1.0]), ("gaussian", [0.6]), ("matern", [1.0]), ("matern", [0.7]), ("expsinesquared", [1.0, 1.0]),
               ("expsinesquared", [0.8, 1.3]), ("rationalquadratic", [1.0, 1.0]), ("rationalquadratic", [0.7, 2.5]),
               ("dotproduct", [1.0]), ("dotproduct", [0.3]), ("pairwisekernel", [0.0])]
OUTER_IDS = [f"{o}-{'-'.join(str(v) for v in h)}" for o, h in OUTER_CASES]


def _bound_doc():
    """How every ABI bound in this file is built.

    A computed sum of terms x_t, each reaching the result through k_t roundings, is within u sum_t k_t |x_t| (+ O(u^2)) of the
    exact sum, u = 2^-53: recursive summation of N terms rounds each partial sum once, so the first term is rounded N - 1 times.
    Both sides are such sums, so the bound of |device - reference| is u (c_dev + c_ref) T_i, T_i the same sum with every factor
    replaced by its magnitude, and c the longest chain of roundings one term can take.  B = A^-1 - alpha alpha^T is formed from
    A^-1 and alpha on both sides, with a rounding relative to |A^-1_jk| + |alpha_j alpha_k|, so T_i takes that in place of |B_jk|:
    at a real shard the two cancel to about 1/sigma^2 and |B| alone would understate the error.

    The weights kappa'(s) and dK/dh depend on s = |f_j - f_k|^2, which both sides compute as a sum of m squares: a weight is
    within C_W ulp of its exact value for the computed s (at most four elementary functions, each within 2 ulp, and the products
    that combine them), plus the propagated error of s, |s w'(s)| (m + 6) u per side (the sum of squares and the sqrt / scaling of
    its root), plus C_Y u |y| w for an exponent e^y whose argument y takes C_Y roundings.  Those two enter as T'_i and T''_i, the
    sums with |s w'(s)| and |y w| in place of |w|."""


@pytest.fixture(scope="module")
def d():
    import dqgp_b200
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")
    return dqgp_b200


def _sp():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _z(P):
    return np.round(np.random.RandomState(5).uniform(0.3, 2.8, P), 4)


def _engine(d, name, **kw):
    enc, ktype, q, layers, dd, n, outer = SHARDS[name]
    x, y = d.synthetic_dataset(n, dd, enc)        # the first rows of every n are the same samples
    if ktype == "projected":
        kw = dict(dict(outer_kernel=outer, training_ignores_outer_kernel=False), **kw)
    return d.AgentEngine(x, y, encoding_type=enc, kernel_type=ktype, num_qubits=q, num_layers=layers, noise_std=SIGMA, rho=100.0,
                         L=100.0, **kw)


def _build_shard(d, name):
    """One analytic step's inputs to the gradient: the full symmetric A^-1 (want_inverse = 2), alpha, the features / states
    and the Jacobian, plus the engine's own gradient."""
    eng = _engine(d, name, gradient="analytic")
    eng.simulate(d.kernels.dev_f64(_z(eng.P)))
    eng.gram()
    eng.factor()
    torch.cuda.synchronize()
    eng.check_info()
    eng.gradient()
    out = dict(Ainv=eng.solver.inverse().clone(), alpha=eng.d_alpha.clone(), F=eng.d_feat[0].clone(), J=eng.d_jac.clone(),
               grad=eng.d_grad.cpu().numpy().copy(), q=eng.q, P=eng.P)
    torch.cuda.synchronize()
    del eng
    return out


@pytest.fixture(scope="module")
def shard(d):
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = _build_shard(d, name)
        return cache[name]
    yield get
    cache.clear()
    torch.cuda.empty_cache()


def _tree_sum(x):
    """Sum over the last dimension in a tree of groups of GROUP: every term takes at most (GROUP - 1) levels roundings."""
    while x.shape[-1] > 1:
        k = x.shape[-1]
        pad = (-k) % GROUP
        if pad:
            x = torch.nn.functional.pad(x, (0, pad))
        x = x.reshape(*x.shape[:-1], -1, GROUP).sum(-1)
    return x[..., 0]


def _levels(n):
    return max(1, math.ceil(math.log(max(n, 2), GROUP) - 1e-12))


def _padded(Ainv, lower_only=False):
    """A^-1 with ld = n + 3 and NaN in the padding columns (and, for the hyper-parameter kernel, above the diagonal)."""
    n = Ainv.shape[0]
    A = torch.full((n, n + 3), float("nan"), dtype=torch.float64, device="cuda")
    A[:, :n] = torch.tril(Ainv) + torch.triu(torch.full_like(Ainv, float("nan")), 1) if lower_only else Ainv
    return A


def _sentinel_out(P):
    """Output buffer of P entries between 4 guard entries on each side, all -7."""
    buf = torch.full((P + 8,), -7.0, dtype=torch.float64, device="cuda")
    return buf, buf[4:4 + P]


def _check_sentinels(buf, P):
    b = buf.cpu().numpy()
    assert np.all(b[:4] == -7.0) and np.all(b[4 + P:] == -7.0), "a write outside the P outputs"
    assert np.all(b[4:4 + P] != -7.0)
    return b[4:4 + P].copy()


# ---- projected kernel ------------------------------------------------------------------------------------------------------------

def _kappa_prime(outer, hyp, s):
    """dkappa/ds of scikit-learn's kernel kappa(s), s = |f - g|^2, in closed form, and the argument of its exponent."""
    if outer == "gaussian":
        g = hyp[0]
        return -g * torch.exp(-g * s), -g * s
    if outer == "matern":                       # (1 + sqrt3 d / l) e^{-sqrt3 d / l}
        y = -math.sqrt(3.0) * torch.sqrt(s) / hyp[0]
        return -1.5 / hyp[0] ** 2 * torch.exp(y), y
    if outer == "expsinesquared":               # e^{-2 sin^2(pi d / p) / l^2}
        l, p = hyp
        dd = torch.sqrt(s.clamp_min(1e-300))
        z = math.pi * dd / p
        y = -2.0 * torch.sin(z) ** 2 / l ** 2
        return -(math.pi / (p * l * l)) * torch.sin(2.0 * z) / dd * torch.exp(y), y
    l, a = hyp                                  # rationalquadratic: (1 + s / (2 a l^2))^-a
    y = -(a + 1.0) * torch.log1p(s / (2.0 * a * l * l))
    return -1.0 / (2.0 * l * l) * torch.exp(y), y


def _projected_reference(outer, hyp, Ainv, alpha, F, J, block=128):
    """grad_i = 1/2 sum_jk B_jk dK_jk/dp_i = 2 sum_j <J_ij, G_j>, G_j = sum_k B_jk kappa'(s_jk) (f_j - f_k) for a stationary
    kernel; the dot product sigma_0^2 + f_j.f_k gives grad_i = sum_j <J_ij, (B F)_j>.  Float64 on the device in blocks of rows,
    the sums over k and over (j, feature) by _tree_sum.  Returns (grad, T, T', T'')."""
    n, m = F.shape
    dot = outer in ("dotproduct", "pairwisekernel")
    G, Ga, Gp, Gy = (torch.empty((n, m), dtype=torch.float64, device=F.device) for _ in range(4))
    aabs = alpha.abs()
    for r0 in range(0, n, block):
        r1 = min(n, r0 + block)
        Bb = Ainv[r0:r1] - alpha[r0:r1, None] * alpha[None, :]
        Ba = Ainv[r0:r1].abs() + aabs[r0:r1, None] * aabs[None, :]
        if dot:
            G[r0:r1] = _tree_sum((Bb[:, :, None] * F[None]).transpose(1, 2).contiguous())
            Ga[r0:r1] = Ba @ F.abs()
            Gp[r0:r1] = 0.0
            Gy[r0:r1] = 0.0
            continue
        D = F[r0:r1, None, :] - F[None, :, :]
        s = (D * D).sum(-1)
        s_ = s.clone().requires_grad_(True)
        w_, _ = _kappa_prime(outer, hyp, s_)
        (dw,) = torch.autograd.grad(w_.sum(), s_)
        w, y = _kappa_prime(outer, hyp, s)
        Da = D.abs()
        G[r0:r1] = _tree_sum(((Bb * w)[:, :, None] * D).transpose(1, 2).contiguous())
        Ga[r0:r1] = ((Ba * w.abs())[:, :, None] * Da).sum(1)
        Gp[r0:r1] = ((Ba * (s * dw).abs().nan_to_num(0.0))[:, :, None] * Da).sum(1)
        Gy[r0:r1] = ((Ba * (w * y).abs())[:, :, None] * Da).sum(1)
        del D, Da, s, s_, w_, dw, w, y
    scale = 1.0 if dot else 2.0
    P = J.shape[0]
    grad = scale * _tree_sum((J * G[None]).reshape(P, -1))
    Ja = J.abs().reshape(P, -1)
    T, Tp, Ty = (scale * (Ja @ X.reshape(-1)) for X in (Ga, Gp, Gy))
    return grad.cpu().numpy(), T.cpu().numpy(), Tp.cpu().numpy(), Ty.cpu().numpy()


def _projected_chains(n, m):
    """(c_dev, c_ref, c_s, c_y) of the projected analytic gradient (_bound_doc).
    Device, per term: f_j - f_k (1), B (2), the weight (C_W), q = b w (1); the running G_j over its segment (seg_cols); the
    segment sum (segments); the contraction, fma per thread over ceil(n m / 256) entries, an 8-level tree, the scale (2).
    Reference: the same per-term roundings plus the product q (f_j - f_k) (1), two trees (over k, and over (j, feature)) and
    the J product and the scale (2)."""
    seg_cols = ((n + GA_SEGMENTS - 1) // GA_SEGMENTS + GA_CHUNK - 1) // GA_CHUNK * GA_CHUNK
    segments = (n + seg_cols - 1) // seg_cols
    term = 1 + 2 + C_W + 1
    c_dev = term + seg_cols + segments + math.ceil(n * m / 256) + 8 + 2
    c_ref = term + 1 + (GROUP - 1) * (_levels(n) + _levels(n * m)) + 2
    return c_dev, c_ref, 2 * (m + 6), 2 * C_Y


def _device_projected(d, outer, hyp, Ainv, alpha, F, J):
    from dqgp_b200 import _lib
    lib = d.load()
    n, m = F.shape
    P = J.shape[0]
    A = _padded(Ainv)
    work = torch.empty(lib.dqgp_grad_analytic_workspace_bytes(n, m) // 8 + 1, dtype=torch.float64, device="cuda")
    buf, grad = _sentinel_out(P)
    rc = lib.dqgp_grad_projected_analytic(_lib.OUTER_KERNELS[outer], _lib.hyp_array(hyp), A.data_ptr(), n + 3, alpha.data_ptr(),
                                          F.data_ptr(), J.data_ptr(), n, m, P, grad.data_ptr(), work.data_ptr(), _sp())
    assert rc == 0, lib.dqgp_last_error()
    torch.cuda.synchronize()
    return _check_sentinels(buf, P)


def _assert_within(got, ref, bound, T, c):
    """|got - ref| <= bound per entry, and the gradient is far above the bound: max |ref| >= 1e3 c u max T."""
    err = np.abs(got - ref)
    assert np.all(err <= bound), (np.max(err / bound), got[np.argmax(err / bound)], ref[np.argmax(err / bound)])
    assert np.abs(ref).max() >= 1e3 * c * U * T.max(), (np.abs(ref).max(), c * U * T.max())


@pytest.mark.parametrize("case", range(len(OUTER_CASES)), ids=OUTER_IDS)
@pytest.mark.parametrize("name", ["cfg4", "cfg5", "cfg4-1025", "cfg5-4099", "cfg4-8193"])
def test_projected_abi_matches_closed_forms(d, shard, name, case):
    """dqgp_grad_projected_analytic on a real shard (ld = n + 3, NaN padding), every outer id at its default and a non-default
    hyper-parameter, against the closed-form reference: |got - ref| <= u (c T + c_s T' + c_y T'') per parameter (_bound_doc,
    _projected_chains; c = 1518 + 100 at n = 8192, m = 30); the gradient is at least 1e3 times that bound's c u T; a second call
    gives the same bits; only the P outputs are written."""
    outer, hyp = OUTER_CASES[case]
    s = shard(name)
    F, J = s["F"], s["J"]
    n, m = F.shape
    got = _device_projected(d, outer, hyp, s["Ainv"], s["alpha"], F, J)
    ref, T, Tp, Ty = _projected_reference(outer, hyp, s["Ainv"], s["alpha"], F, J)
    c_dev, c_ref, c_s, c_y = _projected_chains(n, m)
    c = c_dev + c_ref
    _assert_within(got, ref, U * (c * T + c_s * Tp + c_y * Ty), T, c)
    assert np.array_equal(got, _device_projected(d, outer, hyp, s["Ainv"], s["alpha"], F, J))


def test_projected_reference_is_accurate(d, shard):
    """The float64 reference against the same formulas in np.longdouble at n = 1025 (ExpSineSquared off its defaults: the
    weight with the most elementary functions): within its own share u (c_ref T + c_s T' / 2 + c_y T'' / 2) of the bound, and
    below a tenth of the whole bound the device is held to."""
    outer, hyp = "expsinesquared", [0.8, 1.3]
    s = shard("cfg4-1025")
    F, J = s["F"], s["J"]
    n, m = F.shape
    ref, T, Tp, Ty = _projected_reference(outer, hyp, s["Ainv"], s["alpha"], F, J)
    LD = np.longdouble
    Fl, Jl = F.cpu().numpy().astype(LD), J.cpu().numpy().astype(LD)
    Al, al = s["Ainv"].cpu().numpy().astype(LD), s["alpha"].cpu().numpy().astype(LD)
    l, p = (LD(v) for v in hyp)
    pi = np.arccos(LD(-1))
    G = np.zeros((n, m), dtype=LD)
    for r0 in range(0, n, 64):
        r1 = min(n, r0 + 64)
        D = Fl[r0:r1, None, :] - Fl[None, :, :]
        dd = np.sqrt(np.maximum((D * D).sum(-1), LD(1e-300)))
        z = pi * dd / p
        w = -(pi / (p * l * l)) * np.sin(2 * z) / dd * np.exp(-2 * np.sin(z) ** 2 / (l * l))
        G[r0:r1] = np.einsum("jk,jkl->jl", (Al[r0:r1] - al[r0:r1, None] * al[None, :]) * w, D)
    exact = np.array([2 * np.sum(Jl[i] * G) for i in range(J.shape[0])], dtype=LD)
    c_dev, c_ref, c_s, c_y = _projected_chains(n, m)
    err = np.abs(ref - exact).astype(np.float64)
    assert np.all(err <= U * (c_ref * T + c_s / 2 * Tp + c_y / 2 * Ty))
    assert np.all(err <= 0.1 * U * ((c_dev + c_ref) * T + c_s * Tp + c_y * Ty))


# ---- fidelity kernel -------------------------------------------------------------------------------------------------------------

def _complex(X, dim):
    return torch.view_as_complex(X.reshape(*X.shape[:-1], dim, 2))


def _fidelity_reference(Ainv, alpha, F, J, dim):
    """S = Psi Psi^H, G = (B o S) Psi, grad_i = 2 Re <G, D_i> in complex128 on the device (cuBLAS), the last sum by _tree_sum.
    T_i = 4 sum_j (|B| o |Psi||Psi|^T) |Psi| . |D_i|: moduli in place of the complex values, times 2 because a complex product in
    real arithmetic has at most sqrt 2 times the modulus in absolute terms, twice on a term's path (S, then W Psi)."""
    psi = _complex(F, dim)
    B = Ainv - alpha[:, None] * alpha[None, :]
    G = (B * (psi @ psi.conj().T)) @ psi
    P = J.shape[0]
    grad = np.array([2.0 * _tree_sum((G.conj() * _complex(J[i], dim)).real.reshape(1, -1))[0].item() for i in range(P)])
    pa = psi.abs()
    Ba = Ainv.abs() + alpha.abs()[:, None] * alpha.abs()[None, :]
    Ga = (Ba * (pa @ pa.T)) @ pa
    T = 4.0 * (_complex(J, dim).abs().reshape(P, -1) @ Ga.reshape(-1))
    return grad, T.cpu().numpy()


def _fidelity_chains(n, dim, P):
    """(c_dev, c_ref) of the fidelity analytic gradient (_bound_doc).
    Per-row path (2^q <= 64): s_jk by 2 fma per amplitude (2 dim), B (2), q = b s (1), G_j by 2 fma per column over the
    segment (2 seg_cols), the segment sum (segments), the contraction (ceil(2 n dim / 256) + 8-level tree + scale).
    DMMA path: S over K = 2 dim (2 dim), B o S (3), the GEMM over K = 2 n_pad (2 n_pad), the contraction in GFD_SLICES slices
    (ceil(2 n dim / (slices 256)) + 8) and their sum (1 + 8 + scale).
    Reference: S and W Psi as complex GEMMs (2 dim + 2 n, two real products per complex term), B o S (3), the tree."""
    if dim <= 64:
        seg_cols = ((n + GA_SEGMENTS - 1) // GA_SEGMENTS + GF_CHUNK - 1) // GF_CHUNK * GF_CHUNK
        segments = (n + seg_cols - 1) // seg_cols
        c_dev = 2 * dim + 3 + 2 * seg_cols + segments + math.ceil(2 * n * dim / 256) + 8 + 2
    else:
        npad = (n + GM_BM - 1) // GM_BM * GM_BM
        slices = max(1, min(GFD_SLICES, 2 * npad * npad // P))
        c_dev = 2 * dim + 3 + 2 * npad + math.ceil(2 * n * dim / (slices * 256)) + 8 + 1 + 8 + 2
    c_ref = 2 * dim + 3 + 2 * n + (GROUP - 1) * _levels(2 * n * dim) + 2
    return c_dev, c_ref


def _device_fidelity(d, Ainv, alpha, F, J, dim):
    lib = d.load()
    n = F.shape[0]
    P = J.shape[0]
    A = _padded(Ainv)
    work = torch.empty(lib.dqgp_grad_fidelity_analytic_workspace_bytes(n, dim) // 8 + 2, dtype=torch.float64, device="cuda")
    buf, grad = _sentinel_out(P)
    rc = lib.dqgp_grad_fidelity_analytic(A.data_ptr(), n + 3, alpha.data_ptr(), F.data_ptr(), J.data_ptr(), n, dim, P,
                                         grad.data_ptr(), work.data_ptr(), _sp())
    assert rc == 0, lib.dqgp_last_error()
    torch.cuda.synchronize()
    return _check_sentinels(buf, P)


@pytest.mark.parametrize("name", ["cfg3", "fid-q7-2053", "fid-q10-2053", "fid-q7-8192"])
def test_fidelity_abi_matches_complex_formula(d, shard, name):
    """dqgp_grad_fidelity_analytic on a real shard: config 3 (q = 5, n = 2048: 16 segments of 8 chunks on the per-row path), and
    the DMMA path at q = 7 and 10 with n = 2053 (n_pad = 2176) and at q = 7 with n = 8192 (a GEMM over K = 16384), against the
    complex128 formula: |got - ref| <= (c_dev + c_ref) u T per parameter (_fidelity_chains), the gradient at least 1e3 times
    that, a second call gives the same bits, only the P outputs are written."""
    s = shard(name)
    dim = 1 << s["q"]
    F, J = s["F"], s["J"]
    n, P = F.shape[0], J.shape[0]
    got = _device_fidelity(d, s["Ainv"], s["alpha"], F, J, dim)
    ref, T = _fidelity_reference(s["Ainv"], s["alpha"], F, J, dim)
    c = sum(_fidelity_chains(n, dim, P))
    _assert_within(got, ref, c * U * T, T, c)
    assert np.array_equal(got, _device_fidelity(d, s["Ainv"], s["alpha"], F, J, dim))


def test_fidelity_reference_is_accurate(d, shard):
    """The complex128 reference against G_j = sum_k B_jk <psi_k|psi_j> psi_k in np.longdouble (real and imaginary parts apart)
    at config 3's n = 2048, 2^q = 32: within its own share c_ref u T and below a tenth of the whole bound."""
    s = shard("cfg3")
    dim = 1 << s["q"]
    F, J = s["F"], s["J"]
    n, P = F.shape[0], J.shape[0]
    ref, T = _fidelity_reference(s["Ainv"], s["alpha"], F, J, dim)
    LD = np.longdouble
    X = F.cpu().numpy().astype(LD).reshape(n, dim, 2)
    pr, pi_ = X[..., 0], X[..., 1]
    al = s["alpha"].cpu().numpy().astype(LD)
    B = s["Ainv"].cpu().numpy().astype(LD) - np.outer(al, al)
    Sr, Si = pr @ pr.T + pi_ @ pi_.T, pi_ @ pr.T - pr @ pi_.T          # S_jk = sum_a psi_ja conj(psi_ka)
    Wr, Wi = B * Sr, B * Si
    Gr, Gi = Wr @ pr - Wi @ pi_, Wr @ pi_ + Wi @ pr
    D = J.cpu().numpy().astype(LD).reshape(P, n, dim, 2)
    exact = np.array([2 * np.sum(Gr * D[i, ..., 0] + Gi * D[i, ..., 1]) for i in range(P)], dtype=LD)
    c_dev, c_ref = _fidelity_chains(n, dim, P)
    err = np.abs(ref - exact).astype(np.float64)
    assert np.all(err <= c_ref * U * T)
    assert np.all(err <= 0.1 * (c_dev + c_ref) * U * T)


# ---- hyper-parameters and noise level --------------------------------------------------------------------------------------------

def _hyper_terms(outer, hyp, s):
    """[dK/dh_t] of scikit-learn's kernel in closed form (h_hyp order), and the argument of its exponent."""
    if outer == "gaussian":
        g = hyp[0]
        return [-s * torch.exp(-g * s)], -g * s
    if outer == "matern":
        l = hyp[0]
        y = -math.sqrt(3.0) * torch.sqrt(s) / l
        return [3.0 * s / l ** 3 * torch.exp(y)], y
    if outer == "expsinesquared":
        l, p = hyp
        dd = torch.sqrt(s)
        z = math.pi * dd / p
        y = -2.0 * torch.sin(z) ** 2 / l ** 2
        K = torch.exp(y)
        return [4.0 * torch.sin(z) ** 2 / l ** 3 * K, 4.0 * math.pi * dd * torch.sin(z) * torch.cos(z) / (l * l * p * p) * K], y
    if outer == "rationalquadratic":
        l, a = hyp
        u = s / (2.0 * a * l * l)
        y = -a * torch.log1p(u)
        K = torch.exp(y)
        return [K * (s / l ** 3) / (1.0 + u), K * (u / (1.0 + u) - torch.log1p(u))], y
    return [torch.full_like(s, 2.0 * hyp[0])], torch.zeros_like(s)      # dotproduct sigma_0^2 + f.g


def _hyper_reference(outer, hyp, Ainv, alpha, F, block=256):
    """1/2 sum_jk B_jk dK_jk/dh with s = |f_j - f_k|^2 by direct differences, float64 on the device, in row blocks; per
    hyper-parameter (ref, T, T_s, T_y): T_s = 1/2 sum |B| |d(dK/dh)/ds| (|f_j|^2 + |f_k|^2), the weight of the device's error in
    s (the Gram identity and its snap to zero), T_y = 1/2 sum |B| |y dK/dh|."""
    n, m = F.shape
    k = 1 if outer in ("gaussian", "matern", "dotproduct") else 2
    parts = [[[] for _ in range(4)] for _ in range(k)]
    nrm = (F * F).sum(1)
    aabs = alpha.abs()
    for r0 in range(0, n, block):
        r1 = min(n, r0 + block)
        Bb = Ainv[r0:r1] - alpha[r0:r1, None] * alpha[None, :]
        Ba = Ainv[r0:r1].abs() + aabs[r0:r1, None] * aabs[None, :]
        D = F[r0:r1, None, :] - F[None, :, :]
        s = (D * D).sum(-1)
        del D
        ws, y = _hyper_terms(outer, hyp, s)
        s_ = s.clone().requires_grad_(True)
        ws_, _ = _hyper_terms(outer, hyp, s_.clamp_min(1e-300))
        nsum = nrm[r0:r1, None] + nrm[None, :]
        for t in range(k):
            if ws_[t].requires_grad:
                (dw,) = torch.autograd.grad(ws_[t].sum(), s_, retain_graph=t + 1 < k)
            else:
                dw = torch.zeros_like(s)            # the dot product's dK/dsigma_0 does not depend on s
            parts[t][0].append(_tree_sum((Bb * ws[t]).reshape(1, -1)))
            parts[t][1].append((Ba * ws[t].abs()).sum().reshape(1))
            parts[t][2].append((Ba * dw.abs().nan_to_num(0.0) * nsum).sum().reshape(1))
            parts[t][3].append((Ba * (ws[t] * y).abs()).sum().reshape(1))
    out = []
    for t in range(k):
        ref = 0.5 * _tree_sum(torch.cat(parts[t][0]).reshape(1, -1))[0].item()
        out.append((ref, *(0.5 * torch.cat(parts[t][i]).sum().item() for i in (1, 2, 3))))
    return out


def _hyper_chains(n, m):
    """(c_dev, c_ref, c_s, c_y) of the hyper-parameter gradient (_bound_doc).
    Device: B and its factor 2 (2), the term (C_W), fma over a thread's 16 tile entries, a 5-level warp sum, 8 warps, c_0 (1),
    then grad_reduce_kernel over ceil(tiles / 256) per thread, an 8-level tree and 1/2 (exact).  Reference: B (2), the term
    (C_W), the tree over its n / block row blocks' trees of block n entries.  s: the device forms it by the Gram identity,
    -d^2 = 2 f.g - |f|^2 - |g|^2, whose 2m + 2 terms add to at most 2 (|f|^2 + |g|^2), and snaps it to 0 below 4e-15 (|f|^2 +
    |g|^2): c_s = 2 (m + 2) + 4e-15 / u, plus m + 2 for the reference's s."""
    tiles = ((n + 63) // 64) * ((n + 63) // 64 + 1) // 2
    c_dev = 2 + C_W + 16 + 5 + 8 + 1 + math.ceil(tiles / 256) + 8
    c_ref = 2 + C_W + (GROUP - 1) * (_levels(256 * n) + _levels(n // 256 + 1))
    return c_dev, c_ref, 2 * (m + 2) + 4e-15 / U + m + 2, 2 * C_Y


def _device_hyper(d, outer, hyp, Ainv, alpha, F, k):
    from dqgp_b200 import _lib
    lib = d.load()
    n, m = F.shape
    A = _padded(Ainv, lower_only=True)
    work = torch.empty(lib.dqgp_grad_outer_hyperparameters_workspace_bytes(n) // 8 + 1, dtype=torch.float64, device="cuda")
    buf, grad = _sentinel_out(k + 1)
    rc = lib.dqgp_grad_outer_hyperparameters(_lib.OUTER_KERNELS[outer], _lib.hyp_array(hyp), A.data_ptr(), n + 3, alpha.data_ptr(),
                                             F.data_ptr(), n, m, grad.data_ptr(), work.data_ptr(), _sp())
    assert rc == 0, lib.dqgp_last_error()
    rc = lib.dqgp_grad_noise_std(A.data_ptr(), n + 3, alpha.data_ptr(), n, SIGMA, grad[k:].data_ptr(), _sp())
    assert rc == 0, lib.dqgp_last_error()
    torch.cuda.synchronize()
    return _check_sentinels(buf, k + 1)


HYPER_CASES = [c for c in OUTER_CASES if c[0] != "pairwisekernel"]


@pytest.mark.parametrize("case", range(len(HYPER_CASES)), ids=[OUTER_IDS[OUTER_CASES.index(c)] for c in HYPER_CASES])
@pytest.mark.parametrize("name", ["cfg4", "cfg5"])
def test_hyper_abi_matches_closed_forms(d, shard, name, case):
    """dqgp_grad_outer_hyperparameters + dqgp_grad_noise_std at n = 8192 (8256 lower 64 x 64 tiles) on a real A^-1 with NaN above
    the diagonal (what want_inverse = 1 leaves) and in the padding, on the shard's features with four exact duplicate rows (the
    snap-to-zero and diagonal rules): each dNLL/dh within u (c T + c_s T_s + c_y T_y) of 1/2 sum B o dK/dh (_hyper_chains);
    dNLL/dsigma within (ceil(n / 256) + 8 + 3 + tree) u sigma sum(|A^-1_jj| + alpha_j^2) of sigma tr(B); the gradient at least
    1e3 times c u T; a second call gives the same bits; only the outputs are written."""
    outer, hyp = HYPER_CASES[case]
    s = shard(name)
    F = s["F"].clone()
    n, m = F.shape
    for dst, src in [(1, 0), (2, 0), (4096, 77), (n - 1, 8000)]:
        F[dst] = F[src]
    Ainv = torch.tril(s["Ainv"]) + torch.tril(s["Ainv"], -1).T       # the symmetric matrix the lower triangle describes
    ref = _hyper_reference(outer, hyp, Ainv, s["alpha"], F)
    k = len(ref)
    got = _device_hyper(d, outer, hyp, s["Ainv"], s["alpha"], F, k)
    c_dev, c_ref, c_s, c_y = _hyper_chains(n, m)
    c = c_dev + c_ref
    r, T, Ts, Ty = (np.array(v) for v in zip(*ref))
    _assert_within(got[:k], r, U * (c * T + c_s * Ts + c_y * Ty), T, c)
    diag = torch.diagonal(s["Ainv"])
    a2 = s["alpha"] * s["alpha"]
    noise_ref = SIGMA * _tree_sum((diag - a2).reshape(1, -1))[0].item()
    noise_T = SIGMA * (diag.abs() + a2).sum().item()
    c_noise = 2 + math.ceil(n / 256) + 8 + 1 + 2 + (GROUP - 1) * _levels(n) + 1
    assert abs(got[k] - noise_ref) <= c_noise * U * noise_T
    assert abs(noise_ref) >= 1e3 * c_noise * U * noise_T
    assert np.array_equal(got, _device_hyper(d, outer, hyp, s["Ainv"], s["alpha"], F, k))


def test_hyper_reference_is_accurate(d, shard):
    """The float64 reference of the two RationalQuadratic derivatives (log1p, a power and a quotient: the longest term) against
    np.longdouble on the first 1025 samples of config 4: within its share u (c_ref T + c_s T_s / 3 + c_y T_y / 2) and below a
    tenth of the whole bound."""
    outer, hyp = "rationalquadratic", [0.7, 2.5]
    s = shard("cfg4-1025")
    F, Ainv, alpha = s["F"], s["Ainv"], s["alpha"]
    n, m = F.shape
    ref = _hyper_reference(outer, hyp, Ainv, alpha, F)
    LD = np.longdouble
    Fl = F.cpu().numpy().astype(LD)
    al = alpha.cpu().numpy().astype(LD)
    B = Ainv.cpu().numpy().astype(LD) - np.outer(al, al)
    D = Fl[:, None, :] - Fl[None, :, :]
    sl = (D * D).sum(-1)
    del D
    l, a = LD(hyp[0]), LD(hyp[1])
    u = sl / (2 * a * l * l)
    K = np.exp(-a * np.log1p(u))
    exact = [LD(0.5) * np.sum(B * K * (sl / l ** 3) / (1 + u)), LD(0.5) * np.sum(B * K * (u / (1 + u) - np.log1p(u)))]
    c_dev, c_ref, c_s, c_y = _hyper_chains(n, m)
    for (r, T, Ts, Ty), e in zip(ref, exact):
        err = float(abs(LD(r) - e))
        assert err <= U * (c_ref * T + c_s / 3 * Ts + c_y / 2 * Ty)
        assert err <= 0.1 * U * ((c_dev + c_ref) * T + c_s * Ts + c_y * Ty)


# ---- engine: analytic against extrapolated central differences -------------------------------------------------------------------

def _richardson_check(a, g, h, eps):
    """a: the analytic values; g: central differences at steps h, h/2, h/4; eps(step): a bound on the rounding part of a central
    difference at that step.  With g(t) = a + c2 t^2 + c4 t^4 + ..., R(t) = (4 g(t/2) - g(t)) / 3 = a - c4 t^4 / 4 + O(t^6), so
    R(h) - R(h/2) = 15/16 of R(h)'s h^4 term and |R(h/2) - a| ~ |R(h) - R(h/2)| / 15.  Asserted: |R(h/2) - a| <= 2 |R(h) -
    R(h/2)| / 15 + (4 eps(h/4) + eps(h/2)) / 3 (the 2 leaves the O(t^6) term up to half of the t^4 term), and the rate: the
    second-order error |g(t) - a| shrinks by 4 (1 +- 1/8) from t to t/2 on every parameter where it stands above the rounding
    (16 eps(t)): an analytic value off by delta would pull that ratio to 1 once delta nears the c2 t^2 / 8 of the finest step."""
    g1, g2, g4 = g
    R1, R2 = (4 * g2 - g1) / 3, (4 * g4 - g2) / 3
    tol = 2 * np.abs(R1 - R2) / 15 + (4 * eps(h / 4) + eps(h / 2)) / 3
    assert np.all(np.abs(R2 - a) <= tol), (np.max(np.abs(R2 - a) / tol), a, R2)
    for (ga, gb), t in [((g1, g2), h), ((g2, g4), h / 2)]:
        ea, eb = np.abs(ga - a), np.abs(gb - a)
        live = eb > 16 * eps(t / 2)
        assert live.sum() >= max(1, len(a) // 4), (live.sum(), len(a))
        ratio = ea[live] / eb[live]
        assert np.all(np.abs(ratio - 4.0) <= 0.5), ratio


@pytest.mark.parametrize("name", ["cfg3", "cfg4", "cfg5"])
def test_engine_analytic_gradient_is_the_limit_of_central_differences(d, shard, name):
    """AgentEngine(gradient="analytic") at configs 3, 4 and 5's full shard against AgentEngine(gradient="central_difference",
    shift_value=t) at t = 0.08, 0.04, 0.02 on the same z (_richardson_check).  Rounding part of the central difference:
    tests/test_gpu_fullsize.py pins that path to 1e-8 max |g| at t = pi/8, and rounding scales with 1/t, so eps(t) =
    1e-8 max |g| (pi / 8) / t.  h^4 truncation of R(0.04) with the circuits' unit angle frequencies: ~0.04^4 / 480 of the
    third-derivative scale, far below that."""
    s = shard(name)
    a = s["grad"]
    z = _z(s["P"])
    h = 0.08
    g = []
    for t in (h, h / 2, h / 4):
        eng = _engine(d, name, shift_value=t)
        eng.simulate(d.kernels.dev_f64(z))
        eng.gram()
        eng.factor()
        eng.gradient()
        torch.cuda.synchronize()
        eng.check_info()
        g.append(eng.d_grad.cpu().numpy().copy())
        del eng
    scale = np.abs(a).max()
    _richardson_check(a, g, h, lambda t: 1e-8 * scale * (np.pi / 8) / t)


def test_engine_hyper_gradient_is_the_limit_of_nll_differences(d):
    """AgentEngine(hyper_gradient=True) at config 4's full shard with gamma = 0.6 honoured in training: dNLL/dgamma and
    dNLL/dsigma against central differences of the device NLL at steps 0.04, 0.02, 0.01 (_richardson_check).  Rounding part
    of an NLL difference at step t: tests/test_gpu_fullsize.py pins the NLL to 1e-8 |NLL|, so eps(t) = 1e-8 |NLL| / t."""
    z = d.kernels.dev_f64(_z(d.EncodingCircuit("yz_cx", 8, 4, 3).num_parameters))

    def run(gamma, sigma, hyper=False):
        eng = _engine(d, "cfg4", gradient="analytic", outer_kernel_params={"gamma": gamma}, hyper_gradient=hyper)
        eng.noise_std = sigma
        eng.simulate(z)
        eng.gram()
        eng.factor()
        eng.gradient()
        torch.cuda.synchronize()
        eng.check_info()
        out = (float(eng.d_nll[3].item()), eng.hyper_gradient() if hyper else None)
        del eng
        return out

    nll, got = run(0.6, SIGMA, hyper=True)
    h = 0.04
    for name, at in (("gamma", lambda t: (0.6 + t, SIGMA)), ("noise_std", lambda t: (0.6, SIGMA + t))):
        g = []
        for t in (h, h / 2, h / 4):
            g.append(np.array([(run(*at(t))[0] - run(*at(-t))[0]) / (2 * t)]))
        _richardson_check(np.array([got[name]]), g, h, lambda t: 1e-8 * abs(nll) / t)
