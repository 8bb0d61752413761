"""GPU tests of every simulator kernel at production sample counts: several rounds of the grid-stride team loop, against the
per-set kernels on every row and against the NumPy oracle on sampled rows.

Every launcher caps its grid at (SM count) x (resident CTAs per SM), and each kernel then loops over rounds of teams (a lane
group for q <= 8, a CTA for q >= 9, one sample each).  In the last round the dead teams clamp to the last sample and still take
part in the team's syncs.  The sizing below guarantees at least two full rounds and a ragged last one without asking the
occupancy calculator: at most max_threads_per_SM / team_threads teams are resident on one SM, so with
n >= 2 x SMs x (that bound) every launch needs more than two rounds.  The capacity of one round is a multiple of the SM count,
which is even on every NVIDIA GPU with more than one SM, and n is odd, so the last round is never full.

Each case runs once under torch.profiler and asserts which simulator kernel ran, so a case cannot silently test a fallback."""
import ctypes as C
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

SENTINEL = -1234.5          # fills the tail past the last output row; no kernel may write it
TAIL = 97                   # doubles of sentinel past the output
RAGGED = 37                 # odd and not a multiple of 32: n is odd, so the last round is partial
ORACLE_BUDGET = 1.5e8       # rows x sets x gates x 2^q of the NumPy oracle per case (about 2 s on one CPU core)


@pytest.fixture(scope="module")
def d():
    import dqgp_b200
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")
    return dqgp_b200


def _sp():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# ---- sizing, buffers, sampling -------------------------------------------------------------------------------------------

def team_threads(q):
    """Threads of one team: a lane group of LPS = min(32, 2^max(q-3, 0)) lanes for q <= 8, a CTA of 2^(q-3) threads above."""
    return min(32, 1 << max(q - 3, 0)) if q <= 8 else 1 << (q - 3)


def scale_size(q, sms, max_threads, units=1):
    """Smallest odd n with units * n > 2 * sms * (resident-team bound), and the full rounds that guarantees.  units = S for the
    per-set kernels, whose teams run over the S * n (set, sample) pairs."""
    per_round = sms * (max_threads // team_threads(q))
    n = -(-2 * per_round // units) + RAGGED
    if n % 2 == 0:
        n += 1
    return n, (units * n) // per_round


def prefilled(shape):
    """(buffer, view): the view of `shape` is NaN, followed by TAIL sentinel doubles."""
    numel = int(np.prod(shape))
    buf = torch.full((numel + TAIL,), float("nan"), dtype=torch.float64, device="cuda")
    buf[numel:] = SENTINEL
    return buf, buf[:numel].view(shape)


def assert_filled(buf, out):
    """Every output entry written (no NaN left), nothing written past the last row."""
    assert not torch.isnan(out).any().item(), "an output row was never written"
    assert torch.all(buf[out.numel():] == SENTINEL).item(), "a kernel wrote past the last output row"


def sample_rows(n, rng):
    """The first 16 rows, the last 64 (they hold the ragged last round) and 48 random ones, sorted and distinct."""
    head, tail = np.arange(min(16, n)), np.arange(max(n - 64, 0), n)
    mid = rng.choice(n, size=min(48, n), replace=False)
    return np.unique(np.concatenate([head, tail, mid]))


def oracle_plan(rows, S, P, n_gates, q):
    """Which (rows, sets) the NumPy oracle checks within ORACLE_BUDGET.  All sets on all sampled rows when affordable; else all
    sets on as many sampled rows as fit (a quarter from the head, the rest from the tail, which holds the ragged round); if not
    even 8 rows fit, the base set and the two shifted sets of a few evenly spaced parameters on 8 rows.  The rows left out are
    still compared, device against device, with the per-set kernels."""
    unit = n_gates * (1 << q)
    sets = np.arange(S)
    fit = int(ORACLE_BUDGET // (S * unit))
    if fit >= len(rows):
        return rows, sets
    k = max(fit, 8)
    sub = np.unique(np.concatenate([rows[:k // 4], rows[len(rows) - (k - k // 4):]]))
    if fit >= 8 or P == 0:
        return sub, sets
    n_par = max(1, min(P, int(ORACLE_BUDGET // (len(sub) * 2 * unit))))
    par = np.unique(np.linspace(0, P - 1, n_par).round().astype(int))
    return sub, np.concatenate([[0], 1 + 2 * par, 2 + 2 * par])


def oracle_outputs(gates, q, x, pm, rows, sets, want_states):
    """Oracle states / Pauli features for every (set, row) of the plan: (len(sets), len(rows), ...).  The sets are simulated
    together: the oracle's gate angles broadcast a per-row parameter vector (P, N) like a single one."""
    from oracle import statevector
    xs = x[rows]
    nr = len(rows)
    out = []
    chunk = max(1, (1 << 22) // ((1 << q) * nr))            # at most 4M amplitudes per oracle batch
    for c0 in range(0, len(sets), chunk):
        ss = sets[c0:c0 + chunk]
        X = np.tile(xs, (len(ss), 1))
        Pr = np.repeat(pm[ss], nr, axis=0).T
        psi = statevector.simulate(gates, q, X, Pr)
        v = psi if want_states else statevector.pauli_features(psi, q)
        out.append(v.reshape((len(ss), nr) + v.shape[1:]))
    return np.concatenate(out)


def sim_kernels(fn):
    """Names (with template arguments, no spaces) of the simulator kernels fn launches."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    found = set()
    for e in prof.events():
        m = re.search(r"(statevec_\w*kernel)<([^>]*)>", e.name)
        if m:
            args = m.group(2).replace(" ", "").replace("(bool)0", "false").replace("(bool)1", "true")
            found.add(f"{m.group(1)}<{args}>")
    return found


def _inputs(rng, enc, n, dd):
    lo, hi = (-0.99, 0.99) if enc in ("chebyshev", "kyriienko") else (-2.0, 2.0)
    return rng.uniform(lo, hi, (n, dd))


def _shifted_sets(rng, P):
    from oracle import agent_step
    return agent_step.shifted_parameter_sets(np.round(rng.uniform(-0.5, 3.5, P), 4), np.pi / 8)


def _props():
    p = torch.cuda.get_device_properties(0)
    return p.multi_processor_count, p.max_threads_per_multi_processor


def _call_shifted(lib, ec, want_states, dx, n, dpm, P, out):
    fn = lib.dqgp_states_shifted if want_states else lib.dqgp_features_shifted
    rc = fn(ec.handle, dx.data_ptr(), n, dpm.data_ptr(), P, out.data_ptr(), _sp())
    assert rc == 0, lib.dqgp_last_error()


def _call_per_set(lib, ec, want_states, dx, n, dpm, S, out):
    fn = lib.dqgp_states if want_states else lib.dqgp_features
    rc = fn(ec.handle, dx.data_ptr(), n, dpm.data_ptr(), S, out.data_ptr(), _sp())
    assert rc == 0, lib.dqgp_last_error()


def _shape(q, want_states, *lead):
    return tuple(lead) + ((1 << q, 2) if want_states else (3 * q,))


def _as_complex(t):
    a = t.cpu().numpy()
    return a[..., 0] + 1j * a[..., 1]


# ---- prefix-sharing kernels (dqgp_features_shifted / dqgp_states_shifted) --------------------------------------------------

# (encoding, q, features, layers, states?, DQGP_SV_NO_LC, kernel reached, comparison with the per-set kernels)
SHIFTED = [
    # CX-free plan (yz_cx, kyriienko): the fused-epilogue kernel; team = 1 lane, 4 lanes, a warp, a CTA with paired forks
    ("yz_cx", 3, 2, 2, False, False, "statevec_lc2_kernel<3>", "lc"),
    ("kyriienko", 5, 3, 2, False, False, "statevec_lc2_kernel<5>", "lc"),
    ("yz_cx", 8, 4, 2, False, False, "statevec_lc2_kernel<8>", "lc"),
    ("yz_cx", 9, 3, 2, False, False, "statevec_lc2_kernel<9>", "lc"),
    ("kyriienko", 10, 6, 4, False, False, "statevec_lc2_kernel<10>", "lc"),          # config 5
    # q = 12: four 64 KB state copies do not fit in 227 KB, so lc2 gives way.  With one layer the one-fork kernel's three copies
    # and the gate list fit; with seven layers (413 gates) they do not and the two-fork kernel runs.
    ("kyriienko", 12, 6, 1, False, False, "statevec_lc_kernel<12,false,false>", "lc"),
    ("kyriienko", 12, 6, 7, False, False, "statevec_shared_kernel<12,false>", "bits"),
    # circuits with CRZ gates: the one-fork kernel (CRZ parameters keep two forks)
    ("chebyshev", 4, 2, 2, False, False, "statevec_lc_kernel<4,false,false>", "lc"),
    ("hubregtsen", 7, 3, 1, False, False, "statevec_lc_kernel<7,false,false>", "lc"),
    ("hubregtsen", 9, 3, 1, False, False, "statevec_lc_kernel<9,false,false>", "lc"),
    # states form of the one-fork kernel
    ("hubregtsen", 5, 2, 2, True, False, "statevec_lc_kernel<5,true,false>", "lc"),
    ("hubregtsen", 9, 3, 1, True, False, "statevec_lc_kernel<9,true,false>", "lc"),
    # the two-fork kernel (DQGP_SV_NO_LC): bit-identical to the per-set kernels
    ("yz_cx", 6, 3, 2, False, True, "statevec_shared_kernel<6,false>", "bits"),
    ("hubregtsen", 10, 2, 1, True, True, "statevec_shared_kernel<10,true>", "bits"),
]


@pytest.mark.parametrize("enc,q,dd,layers,want_states,no_lc,kernel,compare", SHIFTED)
def test_shared_prefix_kernels_over_several_rounds(d, monkeypatch, enc, q, dd, layers, want_states, no_lc, kernel, compare):
    from oracle import circuits
    sms, max_threads = _props()
    n, rounds = scale_size(q, sms, max_threads)
    print(f"\n{kernel}: {enc} q={q} L={layers} n={n}, >= {rounds} full rounds + a ragged one")
    rng = np.random.default_rng(1000 * q + 10 * layers + dd)
    x = _inputs(rng, enc, n, dd)
    ec = d.EncodingCircuit(enc, q, dd, layers)
    P = ec.num_parameters
    pm = _shifted_sets(rng, P)
    S = 2 * P + 1
    lib = d.load()
    dx, dpm = d.kernels.dev_f64(x), d.kernels.dev_f64(pm)
    if no_lc:
        monkeypatch.setenv("DQGP_SV_NO_LC", "1")
    buf, out = prefilled(_shape(q, want_states, S, n))
    assert sim_kernels(lambda: _call_shifted(lib, ec, want_states, dx, n, dpm, P, out)) == {kernel}
    assert_filled(buf, out)

    # every row against the per-set kernels
    ref = torch.empty_like(out)
    _call_per_set(lib, ec, want_states, dx, n, dpm, S, ref)
    torch.cuda.synchronize()
    if compare == "bits":
        assert torch.equal(out, ref)
    else:
        assert (out - ref).abs().max().item() <= 2e-14
        if want_states:
            assert torch.equal(out[0], ref[0])                    # the base set is simulated directly
        else:
            assert (out[0] - ref[0]).abs().max().item() <= 5e-15
    del ref

    # sampled rows against the oracle
    rows = sample_rows(n, rng)
    gates = circuits.build_circuit(enc, q, dd, layers)
    o_rows, o_sets = oracle_plan(rows, S, P, len(gates), q)
    got = out[:, torch.from_numpy(o_rows).cuda()][torch.from_numpy(o_sets).cuda()]
    got = _as_complex(got) if want_states else got.cpu().numpy()
    assert np.abs(got - oracle_outputs(gates, q, x, pm, o_rows, o_sets, want_states)).max() <= 1e-12
    base = out[0, torch.from_numpy(rows).cuda()]
    base = _as_complex(base) if want_states else base.cpu().numpy()
    assert np.abs(base - oracle_outputs(gates, q, x, pm, rows, np.array([0]), want_states)[0]).max() <= 1e-12

    # position independence: the sampled rows on their own, through the same kernel, give the same bits
    monkeypatch.setenv("DQGP_SV_FORCE_SHARED", "1")
    m = len(rows)
    dxs = d.kernels.dev_f64(x[rows])
    buf_s, small = prefilled(_shape(q, want_states, S, m))
    assert sim_kernels(lambda: _call_shifted(lib, ec, want_states, dxs, m, dpm, P, small)) == {kernel}
    assert_filled(buf_s, small)
    assert torch.equal(small, out[:, torch.from_numpy(rows).cuda()])


# ---- per-set kernels (dqgp_features / dqgp_states) ---------------------------------------------------------------------------

PER_SET = [("chebyshev", 2, 2, 2), ("hubregtsen", 6, 3, 2), ("yz_cx", 8, 4, 2), ("kyriienko", 9, 4, 1), ("hubregtsen", 12, 2, 1)]


@pytest.mark.parametrize("want_states", [False, True])
@pytest.mark.parametrize("enc,q,dd,layers", PER_SET)
def test_per_set_kernels_over_several_rounds(d, enc, q, dd, layers, want_states):
    from oracle import circuits
    sms, max_threads = _props()
    S = 3
    n, rounds = scale_size(q, sms, max_threads, units=S)
    kernel = f"statevec_{'kernel' if q <= 8 else 'block_kernel'}<{q},{'true' if want_states else 'false'}>"
    print(f"\n{kernel}: {enc} q={q} S={S} n={n} (S*n={S * n}), >= {rounds} full rounds + a ragged one")
    rng = np.random.default_rng(100 * q + dd + int(want_states))
    x = _inputs(rng, enc, n, dd)
    ec = d.EncodingCircuit(enc, q, dd, layers)
    P = ec.num_parameters
    pm = np.round(rng.uniform(-0.5, 3.5, (S, P)), 4)
    lib = d.load()
    dx, dpm = d.kernels.dev_f64(x), d.kernels.dev_f64(pm)
    buf, out = prefilled(_shape(q, want_states, S, n))
    assert sim_kernels(lambda: _call_per_set(lib, ec, want_states, dx, n, dpm, S, out)) == {kernel}
    assert_filled(buf, out)

    rows = sample_rows(n, rng)
    gates = circuits.build_circuit(enc, q, dd, layers)
    got = out[:, torch.from_numpy(rows).cuda()]
    got = _as_complex(got) if want_states else got.cpu().numpy()
    assert np.abs(got - oracle_outputs(gates, q, x, pm, rows, np.arange(S), want_states)).max() <= 1e-12

    m = len(rows)
    buf_s, small = prefilled(_shape(q, want_states, S, m))
    assert sim_kernels(lambda: _call_per_set(lib, ec, want_states, d.kernels.dev_f64(x[rows]), m, dpm, S, small)) == {kernel}
    assert_filled(buf_s, small)
    assert torch.equal(small, out[:, torch.from_numpy(rows).cuda()])


# ---- Jacobian form of the one-fork kernel (dqgp_features_jacobian / dqgp_states_jacobian) ----------------------------------

@pytest.mark.parametrize("want_states", [False, True])
@pytest.mark.parametrize("enc,q,dd,layers", [("hubregtsen", 6, 3, 2), ("yz_cx", 10, 2, 1)])
def test_jacobian_kernel_over_several_rounds(d, enc, q, dd, layers, want_states):
    """The base output equals the per-set kernel on every row bit for bit; the derivative equals central differences of the
    per-set kernel (h = 1e-6) on the sampled rows; the base output equals the oracle there."""
    from oracle import circuits
    sms, max_threads = _props()
    n, rounds = scale_size(q, sms, max_threads)
    kernel = f"statevec_lc_kernel<{q},{'true' if want_states else 'false'},true>"
    print(f"\n{kernel}: {enc} q={q} n={n}, >= {rounds} full rounds + a ragged one")
    rng = np.random.default_rng(7 * q + dd + int(want_states))
    x = _inputs(rng, enc, n, dd)
    ec = d.EncodingCircuit(enc, q, dd, layers)
    P = ec.num_parameters
    p = rng.uniform(0.1, 3.0, P)
    lib = d.load()
    dx, dp = d.kernels.dev_f64(x), d.kernels.dev_f64(p)
    fn = lib.dqgp_states_jacobian if want_states else lib.dqgp_features_jacobian

    def run(dxx, m):
        bf, F = prefilled(_shape(q, want_states, m))
        bj, J = prefilled(_shape(q, want_states, P, m))
        found = sim_kernels(lambda: fn(ec.handle, dxx.data_ptr(), m, dp.data_ptr(), F.data_ptr(), J.data_ptr(), _sp()) == 0
                            or pytest.fail(lib.dqgp_last_error().decode()))
        assert found == {kernel}
        assert_filled(bf, F)
        assert_filled(bj, J)
        return F, J

    F, J = run(dx, n)
    base = ec.states(dx, dp.reshape(1, P)) if want_states else ec.features(dx, dp.reshape(1, P))
    assert torch.equal(F, base[0])
    del base

    rows = sample_rows(n, rng)
    drows = torch.from_numpy(rows).cuda()
    dxs = d.kernels.dev_f64(x[rows])
    h = 1e-6
    sets = np.tile(p, (2 * P, 1))
    for i in range(P):
        sets[2 * i, i] += h
        sets[2 * i + 1, i] -= h
    shifted = ec.states(dxs, d.kernels.dev_f64(sets)) if want_states else ec.features(dxs, d.kernels.dev_f64(sets))
    fd = (shifted[0::2] - shifted[1::2]) / (2 * h)
    Js = J[:, drows]
    scale = max(Js.abs().max().item(), 1e-300) if want_states else 1.0
    assert (Js - fd).abs().max().item() < 5e-9 * scale
    assert Js.abs().max().item() > 1e-3

    gates = circuits.build_circuit(enc, q, dd, layers)
    got = F[drows]
    got = _as_complex(got) if want_states else got.cpu().numpy()
    assert np.abs(got - oracle_outputs(gates, q, x, p[None, :], rows, np.array([0]), want_states)[0]).max() <= 1e-12

    Fs, Jsmall = run(dxs, len(rows))
    assert torch.equal(Fs, F[drows])
    assert torch.equal(Jsmall, J[:, drows])


# ---- the dispatch threshold ------------------------------------------------------------------------------------------------

def test_prefix_sharing_dispatch_threshold(d, monkeypatch):
    """q = 6: 4796 samples are 1199 eight-lane teams per warp-sized unit and stay on the per-set kernel; 4800 are 1200 and switch
    to the prefix-sharing kernel.  Both sides agree on the common rows to 2e-14, with no test hook set."""
    monkeypatch.delenv("DQGP_SV_FORCE_SHARED", raising=False)
    monkeypatch.delenv("DQGP_SV_NO_LC", raising=False)
    enc, q, dd, layers = "yz_cx", 6, 3, 2
    rng = np.random.default_rng(4800)
    x = _inputs(rng, enc, 4800, dd)
    ec = d.EncodingCircuit(enc, q, dd, layers)
    P = ec.num_parameters
    pm = _shifted_sets(rng, P)
    S = 2 * P + 1
    lib = d.load()
    dpm = d.kernels.dev_f64(pm)
    outs = {}
    for n, kernel in [(4796, "statevec_kernel<6,false>"), (4800, "statevec_lc2_kernel<6>")]:
        dx = d.kernels.dev_f64(x[:n])
        buf, out = prefilled(_shape(q, False, S, n))
        assert sim_kernels(lambda: _call_shifted(lib, ec, False, dx, n, dpm, P, out)) == {kernel}
        assert_filled(buf, out)
        outs[n] = out
    assert (outs[4796] - outs[4800][:, :4796]).abs().max().item() <= 2e-14


# ---- input edges, every kernel family --------------------------------------------------------------------------------------

ACOS_EDGES = np.array([-1.0, 1.0, 1.0 - 2.0 ** -52, -(1.0 - 2.0 ** -52), 0.0])
ANGLE_EDGES = np.array([1e6, -1e6, 1e6 - 0.5, -999999.75, 12345.678, -3.0 * 2.0 ** 18, 0.0, 5e-324])

# (encoding, q, features, layers, entry point, test hooks, kernel reached)
EDGE_CASES = [
    ("chebyshev", 4, 2, 2, "features_shifted", {"DQGP_SV_FORCE_SHARED": "1"}, "statevec_lc_kernel<4,false,false>"),
    ("chebyshev", 4, 2, 2, "features_shifted", {"DQGP_SV_FORCE_SHARED": "1", "DQGP_SV_NO_LC": "1"}, "statevec_shared_kernel<4,false>"),
    ("chebyshev", 4, 2, 2, "features", {}, "statevec_kernel<4,false>"),
    ("kyriienko", 5, 3, 2, "features_shifted", {"DQGP_SV_FORCE_SHARED": "1"}, "statevec_lc2_kernel<5>"),
    ("kyriienko", 9, 4, 1, "features_shifted", {"DQGP_SV_FORCE_SHARED": "1"}, "statevec_lc2_kernel<9>"),
    ("kyriienko", 9, 4, 1, "states", {}, "statevec_block_kernel<9,true>"),
    ("kyriienko", 6, 3, 2, "features_jacobian", {}, "statevec_lc_kernel<6,false,true>"),
    ("hubregtsen", 5, 2, 2, "states_shifted", {"DQGP_SV_FORCE_SHARED": "1"}, "statevec_lc_kernel<5,true,false>"),
    ("hubregtsen", 9, 3, 1, "features_shifted", {"DQGP_SV_FORCE_SHARED": "1"}, "statevec_lc_kernel<9,false,false>"),
    ("hubregtsen", 9, 3, 1, "states_shifted", {"DQGP_SV_FORCE_SHARED": "1", "DQGP_SV_NO_LC": "1"}, "statevec_shared_kernel<9,true>"),
    ("hubregtsen", 9, 3, 1, "features", {}, "statevec_block_kernel<9,false>"),
    ("yz_cx", 4, 3, 2, "features_shifted", {"DQGP_SV_FORCE_SHARED": "1"}, "statevec_lc2_kernel<4>"),
    ("yz_cx", 9, 3, 2, "features_shifted", {"DQGP_SV_FORCE_SHARED": "1"}, "statevec_lc2_kernel<9>"),
    ("yz_cx", 7, 3, 1, "states", {}, "statevec_kernel<7,true>"),
    ("yz_cx", 10, 2, 1, "states_jacobian", {}, "statevec_lc_kernel<10,true,true>"),
]


def edge_inputs(enc, dd, P, rng):
    """Rows built from the edge values (every value at every feature position, then random mixes) and parameters at the wrap
    edges: 0, the largest double below pi, and values whose +-pi/8 shifts wrap."""
    vals = ACOS_EDGES if enc in ("chebyshev", "kyriienko") else ANGLE_EDGES
    rows = [np.roll(np.resize(vals, dd), k) for k in range(len(vals))] + [np.full(dd, v) for v in vals]
    x = np.vstack(rows + [rng.choice(vals, dd) for _ in range(9)])
    z = np.resize(np.array([0.0, np.nextafter(np.pi, 0.0), np.pi - np.pi / 16, np.pi / 16, 1.0, np.pi / 8]), P)
    return x, z


def edge_tolerance(gates, x, pm):
    """1e-12 + 4 ulp of the largest angle per data-dependent gate: the device may fuse p + c x where NumPy rounds twice."""
    data = [g for g in gates if g.form not in ("", "p")]
    big = max([np.abs(g.angle(x, p)).max() for g in data for p in pm] + [0.0])
    return 1e-12 + 4 * len(data) * np.spacing(big)


@pytest.mark.parametrize("enc,q,dd,layers,entry,hooks,kernel", EDGE_CASES)
def test_input_edges_match_oracle(d, monkeypatch, enc, q, dd, layers, entry, hooks, kernel):
    """arccos encodings at x = -1, 1, +-(1 - 2^-52), 0; angle encodings up to |x| = 1e6 (sincos's large-argument path);
    parameters 0, just below pi and shifts that wrap.  A fast-math sincos or acos does not come near these tolerances."""
    from oracle import agent_step, circuits
    for k, v in hooks.items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(q + dd)
    ec = d.EncodingCircuit(enc, q, dd, layers)
    P = ec.num_parameters
    x, z = edge_inputs(enc, dd, P, rng)
    n = len(x)
    pm = agent_step.shifted_parameter_sets(z, np.pi / 8)
    assert np.any(pm[1::2] < pm[0]) and np.any(pm[2::2] > pm[0])          # some shifts wrap
    gates = circuits.build_circuit(enc, q, dd, layers)
    want_states = entry.startswith("states")
    lib = d.load()
    dx = d.kernels.dev_f64(x)
    if entry.endswith("jacobian"):
        pm = z[None, :]
        buf, out = prefilled(_shape(q, want_states, 1, n))
        bj, J = prefilled(_shape(q, want_states, P, n))
        fn = lib.dqgp_states_jacobian if want_states else lib.dqgp_features_jacobian
        dz = d.kernels.dev_f64(z)
        found = sim_kernels(lambda: fn(ec.handle, dx.data_ptr(), n, dz.data_ptr(), out.data_ptr(), J.data_ptr(), _sp()) == 0
                            or pytest.fail(lib.dqgp_last_error().decode()))
        assert_filled(bj, J)
    else:
        dpm = d.kernels.dev_f64(pm)
        S = len(pm)
        buf, out = prefilled(_shape(q, want_states, S, n))
        call = _call_shifted if entry.endswith("shifted") else _call_per_set
        found = sim_kernels(lambda: call(lib, ec, want_states, dx, n, dpm, P if entry.endswith("shifted") else S, out))
    assert found == {kernel}
    assert_filled(buf, out)
    got = _as_complex(out) if want_states else out.cpu().numpy()
    ref = oracle_outputs(gates, q, x, pm, np.arange(n), np.arange(len(pm)), want_states)
    assert np.abs(got - ref).max() <= edge_tolerance(gates, x, pm)
