"""GPU tests of the fidelity DMMA kernel (csrc/fid.cu) at every supported state size, 2^q amplitudes for q = 1 .. 12, against
references in np.longdouble: the Gram dqgp_gram_fidelity (MODE 0) and the fused central-difference gradient dqgp_grad_fidelity
(MODE 1).  The kernel streams each state in chunks of 32 doubles: a single chunk shorter than 32 for q <= 3, up to 256 chunks at
q = 12, so each q is its own case.  The states are random, normalised and complex with non-zero imaginary parts: a real state
would hide a wrong sign in the Im<psi_k|psi_j> product."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

QS = list(range(1, 13))
SENTINEL = -1234.5
EPS = 2.0 ** -53


@pytest.fixture(scope="module")
def d():
    import dqgp_b200
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")
    return dqgp_b200


def _sp():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def random_states(rng, shape, dim):
    """Normalised complex states, shape + (dim,), every amplitude with a non-zero imaginary part."""
    z = rng.standard_normal(shape + (dim,)) + 1j * (rng.uniform(0.1, 1.0, shape + (dim,)) * rng.choice([-1, 1], shape + (dim,)))
    return z / np.linalg.norm(z, axis=-1, keepdims=True)


def fidelity_reference(a, b):
    """K[j, k] = |<b_k | a_j>|^2 in long double from the real and imaginary parts: Re = ar.br + ai.bi, Im = ai.br - ar.bi."""
    ar, ai = a.real.astype(np.longdouble), a.imag.astype(np.longdouble)
    br, bi = b.real.astype(np.longdouble), b.imag.astype(np.longdouble)
    re = ar @ br.T + ai @ bi.T
    im = ai @ br.T - ar @ bi.T
    return re * re + im * im


def to_device(z):
    """(…, dim) complex -> contiguous (…, dim, 2) float64 on the device (torch allocations are 256-byte aligned)."""
    t = torch.from_numpy(np.ascontiguousarray(np.stack([z.real, z.imag], axis=-1))).cuda()
    assert t.data_ptr() % 16 == 0
    return t


def gram(lib, psi1, n1, psi2, n2, dim):
    """dqgp_gram_fidelity into K (n1, ldk = n2 + 3): NaN in the logical columns, SENTINEL in the three past them."""
    K = torch.full((n1, n2 + 3), SENTINEL, dtype=torch.float64, device="cuda")
    K[:, :n2] = float("nan")
    same = int(psi1.data_ptr() == psi2.data_ptr())
    assert lib.dqgp_gram_fidelity(psi1.data_ptr(), n1, psi2.data_ptr(), n2, dim, K.data_ptr(), n2 + 3, same, _sp()) == 0, \
        lib.dqgp_last_error()
    K = K.cpu().numpy()
    assert np.all(K[:, n2:] == SENTINEL)                    # nothing written past the logical width
    return K[:, :n2]


SHAPES = [(1, 1), (63, 65), (64, 64), (65, 129), (130, 7)]


@pytest.mark.parametrize("q", QS)
def test_gram_fidelity_matches_long_double_reference(d, q):
    """Two state arrays and one array against itself (Psi2 = the first n2 states of Psi1), ragged shapes on both sides of the
    64-state tile, ld = n2 + 3.  Bound: each of the two dot products of 2 * 2^q doubles errs by at most 2 * 2^q * 2^-53 for unit
    states, so |K - K_ref| <= 4 * 2^q * 2^-53."""
    dim = 1 << q
    rng = np.random.default_rng(q)
    A, B = random_states(rng, (130,), dim), random_states(rng, (129,), dim)
    ref_ab, ref_aa = fidelity_reference(A, B), fidelity_reference(A, A)
    dA, dB = to_device(A), to_device(B)
    lib = d.load()
    tol = 4 * dim * EPS
    for n1, n2 in SHAPES:
        K = gram(lib, dA, n1, dB, n2, dim)
        assert np.abs(K - ref_ab[:n1, :n2]).max() <= tol, (n1, n2)
        K = gram(lib, dA, n1, dA, n2, dim)
        assert np.abs(K - ref_aa[:n1, :n2]).max() <= tol, (n1, n2, "same")
    # a NaN amplitude of state j of Psi1 (state k of Psi2) gives NaN in row j (column k) and nowhere else
    j, k = 40, 100
    A[j, rng.integers(dim)] = complex(np.nan, 0.0)
    B[k, dim - 1] = complex(0.0, np.nan)                       # in the last chunk
    K = gram(lib, to_device(A), 65, to_device(B), 129, dim)
    mask = np.zeros((65, 129), dtype=bool)
    mask[j, :] = True
    mask[:, k] = True
    assert np.array_equal(np.isnan(K), mask)
    assert np.abs(K[~mask] - ref_ab[:65, :129][~mask]).max() <= tol


@pytest.mark.parametrize("q", QS)
def test_gram_fidelity_of_basis_states_is_exact(d, q):
    """Computational-basis states with phases 1, -1, i, -i: every entry is exactly 0 or 1."""
    dim = 1 << q
    rng = np.random.default_rng(100 + q)
    lib = d.load()
    n1, n2 = 65, 129
    a, b = rng.integers(dim, size=n1), rng.integers(dim, size=n2)
    phases = np.array([1, -1, 1j, -1j])
    A = np.zeros((n1, dim), dtype=np.complex128)
    B = np.zeros((n2, dim), dtype=np.complex128)
    A[np.arange(n1), a] = phases[rng.integers(4, size=n1)]
    B[np.arange(n2), b] = phases[rng.integers(4, size=n2)]
    K = gram(lib, to_device(A), n1, to_device(B), n2, dim)
    assert np.array_equal(K, (a[:, None] == b[None, :]).astype(np.float64))


def _tiles_ainv(rng, n, ld):
    """A symmetric matrix M (n x n) and A^-1 as passed: (n, ld) holding M in the lower 128 x 128 tiles and NaN in the tiles
    above them and in the padding columns, which the gradient must never read."""
    M = rng.standard_normal((n, n))
    M = M + M.T
    A = np.full((n, ld), np.nan)
    r, c = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    lower = (r // 128) >= (c // 128)
    A[:, :n][lower] = M[lower]
    return M, A


@pytest.mark.parametrize("q", QS)
def test_grad_fidelity_matches_materialised_central_difference(d, q):
    """grad_i = 1/2 sum_jk B_jk (K+_i - K-_i)_kj / (2h), B = M - alpha alpha^T, with the shifted Grams in long double, for
    P = 1, 2, 3 (the per-parameter partials are double-buffered) and n on both sides of the 64- and 128-state tiles.
    Bound: each K entry errs by at most 4 * 2^q * 2^-53 (see the Gram test), so K+ - K- by 8 * 2^q * 2^-53; the fixed-order
    reduction of the weighted terms (|K+ - K-| <= 1) adds at most 64 * 2^-53 sum|B|:
        |grad - ref| <= (8 * 2^q + 64) * 2^-53 * sum|B| / 2 / (2h).
    A second call gives the same bits."""
    dim = 1 << q
    rng = np.random.default_rng(200 + q)
    lib = d.load()
    h = np.pi / 8
    ns = [1, 63, 130] if q < 10 else [1, 65, 129]
    n_max, P_max = ns[-1], 3
    pool = random_states(rng, (2 * P_max + 1, n_max), dim)
    Ks = [fidelity_reference(pool[s], pool[s]) for s in range(1, 2 * P_max + 1)]       # sets 1 .. 2P (set 0 is not read)
    for n in ns:
        ld = n + 5
        M, A = _tiles_ainv(rng, n, ld)
        alpha = rng.standard_normal(n)
        B = M - np.outer(alpha, alpha)
        dA, dal = torch.from_numpy(A).cuda(), torch.from_numpy(alpha).cuda()
        for P in (1, 2, 3):
            psi = to_device(pool[:2 * P + 1, :n])
            work = torch.empty(lib.dqgp_grad_workspace_bytes(n, P) // 8 + 1, dtype=torch.float64, device="cuda")
            grads = []
            for _ in range(2):
                g = torch.full((P,), np.nan, dtype=torch.float64, device="cuda")
                assert lib.dqgp_grad_fidelity(dA.data_ptr(), ld, dal.data_ptr(), psi.data_ptr(), n, dim, P, h, g.data_ptr(),
                                              work.data_ptr(), _sp()) == 0, lib.dqgp_last_error()
                grads.append(g.cpu().numpy())
            assert np.array_equal(grads[0], grads[1])
            Bl = B.astype(np.longdouble)
            ref = np.array([float(0.5 * np.sum(Bl * (Ks[2 * i][:n, :n] - Ks[2 * i + 1][:n, :n]).T) / (2 * h)) for i in range(P)])
            tol = (8 * dim + 64) * EPS * np.abs(B).sum() / 2 / (2 * h)
            assert np.all(np.abs(grads[0] - ref) <= tol), (n, P, grads[0], ref, tol)
