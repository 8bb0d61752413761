"""Device-resident engines: one agent's step (``AgentEngine``) and the multi-agent ADMM iteration over the
GPUs of a node (``AdmmEngine``).

``AgentEngine.step`` is the GPU equivalent of ``RiemannianAgent.train_and_update``
(``agent_riemannian.py:314-491``): 2P+1 parameter sets -> statevector features/states for all sets ->
unshifted Gram written straight into the solver's padded matrix -> + sigma^2 I -> blocked Cholesky, alpha,
explicit inverse, logdet -> fused central-difference gradient (no shifted Gram is materialised) -> NLL terms
-> local ADMM update.  Everything is enqueued on the current CUDA stream; nothing syncs with the host.

``AdmmEngine.iteration`` is the body of the driver loop (``main.py:2507-2555``) minus CV and printing:
consensus z from all agents' (theta, psi), then every local agent's step; with several ranks
(``torch.distributed``, one process per GPU) the only exchange is an all-gather of the (A, P) theta/psi
rows — a few KB over NVLink.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import OUTER_KERNELS, DqgpError, check
from .kernels import EncodingCircuit, _require_cuda, dev_f64, outer_hyp, stream_ptr

PERIOD = float(np.pi)
HYPER_NAMES = {"gaussian": ("gamma",), "matern": ("length_scale",), "expsinesquared": ("length_scale", "periodicity"),
               "rationalquadratic": ("length_scale", "alpha"), "dotproduct": ("sigma_0",), "pairwisekernel": ()}


class _DeviceMatrix:
    """Zero-copy view of library-owned device memory as a torch tensor (tests / diagnostics)."""

    def __init__(self, ptr, shape, strides_bytes):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": "<f8", "data": (int(ptr), False),
                                         "version": 2, "strides": strides_bytes}


class Solver:
    """``dqgp_solver`` handle: padded fp64 workspace + task tables for Cholesky / inverse / solve."""

    def __init__(self, n, outer_blocks=0, lean=False):
        """``lean``: one padded square instead of three (factor in place, inverted diagonal blocks, rotating panel
        buffers): no triangular inverse / A^-1, for prediction at sizes where three squares do not fit in HBM."""
        self._lib = _lib.load()
        h = C.c_void_p()
        create = self._lib.dqgp_solver_create_lean if lean else self._lib.dqgp_solver_create_ex
        check(create(int(n), int(outer_blocks), C.byref(h)), "dqgp_solver_create")
        self.handle, self.n, self.lean = h, int(n), bool(lean)
        self.ld = self._lib.dqgp_solver_ld(h)
        self.matrix_ptr = self._lib.dqgp_solver_matrix(h)
        self.inverse_ptr = self._lib.dqgp_solver_inverse(h)
        self.bytes = int(self._lib.dqgp_solver_bytes(h))

    def _view(self, ptr):
        return torch.as_tensor(_DeviceMatrix(ptr, (self.n, self.n), (self.ld * 8, 8)), device="cuda")

    def matrix(self):
        return self._view(self.matrix_ptr)

    def inverse(self):
        return self._view(self.inverse_ptr)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self._lib.dqgp_solver_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class AgentEngine:
    def __init__(self, X, Y, *, encoding_type, kernel_type, num_qubits, num_layers, noise_std, rho, L,
                 outer_kernel="gaussian", shift_value=np.pi / 8, training_ignores_outer_kernel=True, cholesky_outer_blocks=0,
                 gradient="central_difference", outer_kernel_params=None, hyper_gradient=False):
        """``gradient``: "central_difference" = the reference's rule (dK_i = (K(p + h e_i) - K(p - h e_i)) / 2h, h = pi/8,
        agent_riemannian.py:275) - the parity path; "analytic" (opt-in, SURVEY 8(f) row 3) = the exact derivative of the NLL:
        feature Jacobian from one extra suffix simulation per parameter and ONE pass over the n^2 Gram entries.  The analytic
        mode does NOT reproduce the reference's trajectories (its h = pi/8 difference is far from the derivative).  It takes
        every outer kernel of the projected kernel and the fidelity kernel up to 12 qubits.  It keeps the derivative of every
        sample's state (fidelity) or features (projected) for every parameter resident: P * n * 2^q * 16 bytes for the fidelity
        kernel, e.g. 5.4 GB at q = 10, n = 8192, P = 40, plus a workspace of about 16 n^2 bytes from 2^q = 128 on.

        ``outer_kernel_params``: hyper-parameters of the outer kernel in the reference's format ({"gamma": 0.5},
        {"length_scale": 0.7, "periodicity": 1.3}, ...; kernels.outer_hyp), used by the training Gram and both gradient modes.
        None = scikit-learn's defaults.  Only meaningful when the training kernel honours `outer_kernel`: with
        training_ignores_outer_kernel=True (Gaussian, gamma = 1) or the fidelity kernel a value raises ValueError.
        ``hyper_gradient``: every gradient() also computes dNLL/dh for the hyper-parameters h of the outer kernel the training
        Gram uses (the Gaussian's gamma under training_ignores_outer_kernel=True) and dNLL/dsigma for the noise level (a pass over
        the lower tiles of A^-1 and one over its diagonal); read them with `hyper_gradient()`."""
        _require_cuda()
        self._lib = _lib.load()
        X = np.asarray(X, dtype=np.float64)
        X = X.reshape(-1, 1) if X.ndim == 1 else X
        self.n, self.d = X.shape
        if kernel_type not in ("fidelity", "projected"):
            raise ValueError(f"Unknown kernel type: {kernel_type}")
        self.kernel_type = kernel_type
        self.circuit = EncodingCircuit(encoding_type, num_qubits, self.d, num_layers)
        self.q, self.P = int(num_qubits), self.circuit.num_parameters
        self.S = 2 * self.P + 1
        # Q1: the reference's shifted-kernel workers never receive the outer kernel, so training Grams are
        # always Gaussian(gamma=1); training_ignores_outer_kernel=False honours `outer_kernel` instead.
        self.outer_kernel = "gaussian" if training_ignores_outer_kernel else outer_kernel
        if outer_kernel_params is not None and (training_ignores_outer_kernel or kernel_type != "projected"):
            raise ValueError("outer_kernel_params needs kernel_type='projected' and training_ignores_outer_kernel=False: "
                             "otherwise the training kernel is not the outer kernel they parametrise")
        self._outer_id = OUTER_KERNELS[self.outer_kernel] if kernel_type == "projected" else 0
        self._hyp = _lib.hyp_array(outer_hyp(self.outer_kernel, outer_kernel_params)) if kernel_type == "projected" else None
        # scikit-learn's names of the differentiated hyper-parameters, in h_hyp order (PairwiseKernel(metric="linear") has none)
        self.hyper_names = list(HYPER_NAMES[self.outer_kernel]) if kernel_type == "projected" else []
        self.noise_std, self.rho, self.L, self.h = float(noise_std), float(rho), float(L), float(shift_value)
        self.d_X = dev_f64(X)
        self.d_Y = dev_f64(np.asarray(Y, dtype=np.float64).reshape(-1))
        dev = self.d_X.device
        f64 = dict(dtype=torch.float64, device=dev)
        self.m = 3 * self.q if kernel_type == "projected" else 2 * (1 << self.q)   # doubles per sample per set
        if gradient not in ("central_difference", "analytic"):
            raise ValueError(f"Unknown gradient mode: {gradient}")
        self.gradient_mode = gradient
        self.d_Pm = torch.empty((self.S, self.P), **f64)
        if gradient == "analytic":
            self.d_feat = torch.empty((1, self.n, self.m), **f64)
            self.d_jac = torch.empty((self.P, self.n, self.m), **f64)
            wbytes = (self._lib.dqgp_grad_analytic_workspace_bytes(self.n, self.m) if kernel_type == "projected"
                      else self._lib.dqgp_grad_fidelity_analytic_workspace_bytes(self.n, 1 << self.q))
            self.d_work_a = torch.empty(max(1, wbytes // 8), **f64)
        else:
            self.d_feat = torch.empty((self.S, self.n, self.m), **f64)
        self.cholesky_outer_blocks = int(cholesky_outer_blocks)
        self.solver = Solver(self.n, cholesky_outer_blocks)
        self.d_alpha = torch.empty(self.n, **f64)
        self.d_logdet = torch.zeros(1, **f64)
        self.d_info = torch.zeros(1, dtype=torch.int32, device=dev)
        self.d_grad = torch.empty(self.P, **f64)
        self.d_nll = torch.empty(4, **f64)
        self.d_work = torch.empty(max(1, self._lib.dqgp_grad_workspace_bytes(self.n, self.P) // 8), **f64)
        self.hyper_gradient_enabled = bool(hyper_gradient)
        if self.hyper_gradient_enabled:
            # [dNLL/dh in h_hyp order, dNLL/dsigma]
            self.d_hyper_grad = torch.empty(len(self.hyper_names) + 1, **f64)
            self.d_work_h = torch.empty(max(1, self._lib.dqgp_grad_outer_hyperparameters_workspace_bytes(self.n) // 8), **f64)
        self.entries_per_step = self.S * self.n * self.n    # SURVEY §8(d): full squares, all 2P+1 sets
        self.share_prefix = True

    def load_data(self, X, Y, always=False):
        """Refresh the resident shard from host arrays through PERSISTENT pinned staging buffers (allocated once per engine:
        a `pin_memory()` per call is a cudaHostAlloc, which cost 3% of an N=8 iteration in round 1).  The reference re-pickles
        X_i, Y_i to its workers every iteration (main.py:2530-2542); here the shard stays resident on its GPU and is
        re-uploaded only when the host arrays differ from the staged copy (an exact comparison, ~10 us for 8192 x 4) or
        when `always` is set (the bench's e2e leg, whose contract counts the shard's H2D in every step).
        Returns the bytes copied host -> device."""
        if getattr(self, "_h_X", None) is None:
            self._h_X = torch.empty((self.n, self.d), dtype=torch.float64).pin_memory()
            self._h_Y = torch.empty((self.n,), dtype=torch.float64).pin_memory()
            self._h_X_np, self._h_Y_np = self._h_X.numpy(), self._h_Y.numpy()
            self._staged, self._upload_done = False, None
        X = np.asarray(X, dtype=np.float64).reshape(self.n, self.d)
        Y = np.asarray(Y, dtype=np.float64).reshape(-1)
        if self._staged and not always and np.array_equal(X, self._h_X_np) and np.array_equal(Y, self._h_Y_np):
            return 0
        if self._upload_done is not None:
            self._upload_done.synchronize()          # the previous async H2D must have read the staging buffers
        np.copyto(self._h_X_np, X)
        np.copyto(self._h_Y_np, Y)
        self.d_X.copy_(self._h_X, non_blocking=True)
        self.d_Y.copy_(self._h_Y, non_blocking=True)
        self._upload_done = torch.cuda.Event()
        self._upload_done.record()
        self._staged = True
        return X.nbytes + Y.nbytes

    def staging(self):
        """A free (in, out) pair of pinned host buffers for one train_and_update call: (2, P) for z / psi and the packed result
        [theta, psi, nll terms(4), gradient, info].  Pairs are recycled through `release()`; a new pair is allocated only while
        every existing one is in flight."""
        if getattr(self, "_staging_pool", None) is None:
            self._staging_pool = []
        if self._staging_pool:
            return self._staging_pool.pop()
        return (torch.empty((2, self.P), dtype=torch.float64).pin_memory(),
                torch.empty((3 * self.P + 5,), dtype=torch.float64).pin_memory())

    def release(self, pair):
        self._staging_pool.append(pair)

    # -- phases (each enqueues on the current stream) ----------------------------------------------------------
    def simulate(self, d_z, first=0, count=None):
        """Parameter sets (all 2P+1, always) + statevector features/states of sets [first, first+count)."""
        lib, st = self._lib, stream_ptr()
        if first == 0:
            check(lib.dqgp_shift_parameter_sets(d_z.data_ptr(), self.P, self.h, PERIOD, self.d_Pm.data_ptr(), st), "shift sets")
        count = self.S - first if count is None else count
        if self.gradient_mode == "analytic":
            fn = lib.dqgp_features_jacobian if self.kernel_type == "projected" else lib.dqgp_states_jacobian
            check(fn(self.circuit.handle, self.d_X.data_ptr(), self.n, self.d_Pm.data_ptr(), self.d_feat.data_ptr(), self.d_jac.data_ptr(), st),
                  "jacobian")
            return
        if first == 0 and count == self.S and self.share_prefix:
            # all 2P+1 central-difference sets of a sample share the circuit prefix before the shifted gate
            fn = lib.dqgp_features_shifted if self.kernel_type == "projected" else lib.dqgp_states_shifted
            check(fn(self.circuit.handle, self.d_X.data_ptr(), self.n, self.d_Pm.data_ptr(), self.P, self.d_feat.data_ptr(), st),
                  "statevector (shared prefix)")
            return
        fn = lib.dqgp_features if self.kernel_type == "projected" else lib.dqgp_states
        check(fn(self.circuit.handle, self.d_X.data_ptr(), self.n, self.d_Pm[first].data_ptr(), count,
                 self.d_feat[first].data_ptr(), st), "statevector")

    def gram(self, full=False):
        """Unshifted Gram + sigma^2 I into the solver matrix: the lower 64x64 tiles only (all the Cholesky reads), or, for the
        LU fallback, the whole symmetric matrix (`full`)."""
        lib, st, s = self._lib, stream_ptr(), self.solver
        base = self.d_feat.data_ptr()          # set 0 = unshifted parameters
        if self.kernel_type == "projected":
            check(lib.dqgp_gram_projected(self._outer_id, self._hyp, base, self.n, base, self.n, self.m, s.matrix_ptr, s.ld, 1 if full else 2, st),
                  "gram projected")
        else:
            check(lib.dqgp_gram_fidelity(base, self.n, base, self.n, 1 << self.q, s.matrix_ptr, s.ld, 1, st), "gram fidelity")
        check(lib.dqgp_add_diagonal(s.matrix_ptr, self.n, s.ld, self.noise_std ** 2, st), "add diagonal")

    def factor(self):
        # the fused central-difference gradient reads the lower tiles of A^-1; the analytic one its full symmetric image
        check(self._lib.dqgp_potrf_solve_inv(self.solver.handle, self.d_Y.data_ptr(), self.d_alpha.data_ptr(),
                                             self.d_logdet.data_ptr(), self.d_info.data_ptr(), 2 if self.gradient_mode == "analytic" else 1,
                                             stream_ptr()), "potrf")

    def factor_lu(self):
        """The reference's fallback when np.linalg.cholesky raises (agent_riemannian.py:419-425): partial-pivoting LU of
        C + sigma^2 I (needs `gram(full=True)`), alpha and the explicit inverse by the two triangular solves, and
        slogdet for the NLL (:442-444).  A non-positive determinant gives NaN: the reference then takes
        log(det(C + 1e-8 I)) of a non-positive number (:444).  The third rung, np.linalg.pinv (:427-428), is reached in the
        reference only when LAPACK raises on non-finite input; here non-finite input propagates NaN."""
        lib, st, s = self._lib, stream_ptr(), self.solver
        if getattr(self, "d_lu_work", None) is None:
            self.d_lu_work = torch.empty(int(lib.dqgp_lu_workspace_bytes(self.n)) // 8 + 2, dtype=torch.float64, device=self.d_X.device)
            self.d_slogdet = torch.empty(2, dtype=torch.float64, device=self.d_X.device)
        check(lib.dqgp_lu_solve_inv(s.matrix_ptr, s.ld, self.n, self.d_Y.data_ptr(), self.d_alpha.data_ptr(), s.inverse_ptr, s.ld,
                                    self.d_slogdet.data_ptr(), self.d_lu_work.data_ptr(), st), "lu fallback")
        nan = torch.full((), float("nan"), dtype=torch.float64, device=self.d_X.device)
        self.d_logdet.copy_(torch.where(self.d_slogdet[1] > 0, self.d_slogdet[0], nan).reshape(1))
        self.d_info.zero_()
        self.used_lu_fallback = True

    def step_fallback(self, d_z, d_psi, d_theta_out, d_psi_out):
        """Redo a step whose Cholesky failed (`check_info` / d_info > 0) down the reference's ladder: same parameter sets and
        features, full symmetric Gram, LU instead of Cholesky, then the same fused gradient / NLL / local update."""
        self.simulate(d_z)
        self.gram(full=True)
        self.factor_lu()
        self.gradient()
        self.update(d_psi, d_theta_out, d_psi_out)

    def gradient(self):
        lib, st, s = self._lib, stream_ptr(), self.solver
        if self.gradient_mode == "analytic" and self.kernel_type == "fidelity":
            check(lib.dqgp_grad_fidelity_analytic(s.inverse_ptr, s.ld, self.d_alpha.data_ptr(), self.d_feat.data_ptr(), self.d_jac.data_ptr(),
                                                  self.n, 1 << self.q, self.P, self.d_grad.data_ptr(), self.d_work_a.data_ptr(), st),
                  "grad fidelity analytic")
        elif self.gradient_mode == "analytic":
            check(lib.dqgp_grad_projected_analytic(self._outer_id, self._hyp, s.inverse_ptr, s.ld, self.d_alpha.data_ptr(), self.d_feat.data_ptr(),
                                                   self.d_jac.data_ptr(), self.n, self.m, self.P, self.d_grad.data_ptr(),
                                                   self.d_work_a.data_ptr(), st), "grad analytic")
        elif self.kernel_type == "projected":
            check(lib.dqgp_grad_projected(self._outer_id, self._hyp, s.inverse_ptr, s.ld, self.d_alpha.data_ptr(),
                                          self.d_feat.data_ptr(), self.n, self.m, self.P, self.h, self.d_grad.data_ptr(),
                                          self.d_work.data_ptr(), st), "grad projected")
        else:
            check(lib.dqgp_grad_fidelity(s.inverse_ptr, s.ld, self.d_alpha.data_ptr(), self.d_feat.data_ptr(), self.n,
                                         1 << self.q, self.P, self.h, self.d_grad.data_ptr(), self.d_work.data_ptr(), st),
                  "grad fidelity")
        check(lib.dqgp_nll_terms(self.d_logdet.data_ptr(), self.d_Y.data_ptr(), self.d_alpha.data_ptr(), self.n,
                                 self.d_nll.data_ptr(), st), "nll")
        if self.hyper_gradient_enabled:
            k = len(self.hyper_names)
            if k:
                check(lib.dqgp_grad_outer_hyperparameters(self._outer_id, self._hyp, s.inverse_ptr, s.ld, self.d_alpha.data_ptr(),
                                                          self.d_feat.data_ptr(), self.n, self.m, self.d_hyper_grad.data_ptr(),
                                                          self.d_work_h.data_ptr(), st), "grad outer hyper-parameters")
            check(lib.dqgp_grad_noise_std(s.inverse_ptr, s.ld, self.d_alpha.data_ptr(), self.n, self.noise_std,
                                          self.d_hyper_grad[k:].data_ptr(), st), "grad noise_std")

    def hyper_gradient(self):
        """dNLL/dh of the last gradient() (synchronises): {scikit-learn's hyper-parameter name: value} for the hyper-parameters of
        the training Gram's outer kernel (none for the fidelity kernel and PairwiseKernel), plus
        "noise_std": dNLL/dsigma.  Derivatives with respect to log h are h times these."""
        if not self.hyper_gradient_enabled:
            raise ValueError("hyper_gradient() needs AgentEngine(..., hyper_gradient=True)")
        g = self.d_hyper_grad.cpu().numpy()
        return {**{name: float(v) for name, v in zip(self.hyper_names, g)}, "noise_std": float(g[-1])}

    def update(self, d_psi, d_theta_out, d_psi_out):
        # z wrapped to the manifold = row 0 of the parameter-set table (agent_riemannian.py:378)
        check(self._lib.dqgp_admm_local(self.d_Pm.data_ptr(), self.d_grad.data_ptr(), d_psi.data_ptr(), self.P, self.rho, self.L,
                                        PERIOD, d_theta_out.data_ptr(), d_psi_out.data_ptr(), stream_ptr()), "admm local")

    def step(self, d_z, d_psi, d_theta_out, d_psi_out):
        # Overlapping the 2P shifted simulations with the factorisation (side streams at equal or lower priority, before
        # or after the factorisation's launches) was measured three ways and always lost 1-3%: both want the FP64 pipe,
        # and resident simulator CTAs take the register / shared-memory slots of the trailing-update GEMMs.
        self.simulate(d_z)
        self.gram()
        self.factor()
        self.gradient()
        self.update(d_psi, d_theta_out, d_psi_out)

    def launches_per_step(self):
        """Kernel launches of one step() (counted from the launch structure of csrc/chol.cu and friends)."""
        nblk = (self.n + 127) // 128
        levels = int(np.ceil(np.log2(nblk))) if nblk > 1 else 0
        potrf = self._lib.dqgp_solver_potrf_launches(self.solver.handle) + (1 if nblk > 1 else 0)   # + copy of the panels
        pad = 1 + (1 if self.n % 128 else 0)
        hyper = (2 * (len(self.hyper_names) > 0) + 1) if self.hyper_gradient_enabled else 0   # (pass, reduce) noise
        return (2 + 2 + pad + potrf + 2 * levels + 3 + 1        # sets, sim, gram, diag, pad, potrf, trtri, solve, lauum
                + (3 if self.kernel_type == "projected" else 2) + 1 + 1 + hyper)   # (norms) grad reduce, nll, local update

    def check_info(self):
        """Host check of the Cholesky status (syncs).  >0 = index of the first non-positive pivot."""
        info = int(self.d_info.item())
        if info != 0:
            raise np.linalg.LinAlgError(f"Cholesky failed at pivot {info}: K + sigma^2 I is not positive definite")


def synthetic_dataset(n, d, encoding, seed=0):
    """SURVEY §8(d) / BASELINE.md §4 synthetic inputs (identical to oracle.driver.synthetic_dataset)."""
    rng = np.random.default_rng(seed)
    lo, hi = (-0.99, 0.99) if encoding in ("chebyshev", "kyriienko") else (-2.0, 2.0)
    x = rng.uniform(lo, hi, (n, d))
    y = np.sin(x.sum(axis=1)) + 0.1 * rng.standard_normal(n)
    return x, y


def agent_block(rank, world_size, n_agents):
    """Contiguous block of agents owned by `rank`: agent a lives on rank a // (A / world).  The blocks are in
    rank order, so an all-gather of the per-rank (A/world, P) rows reproduces the (A, P) arrays in agent order and
    every rank sums the consensus in the same order as np.sum(axis=0) (riemannian_optimizer.py:42-43)."""
    if n_agents % world_size:
        raise ValueError(f"{n_agents} agents do not split evenly over {world_size} ranks")
    per = n_agents // world_size
    return range(rank * per, (rank + 1) * per)


def exchange_rows(full, local, group=None, world_size=1):
    """The ONLY cross-agent exchange of the path (main.py:2523 / :2550-2555): gather every rank's (A_local, ...) rows
    (theta and psi side by side) into the replicated (A, ...) array.  NCCL over NVLink for CUDA tensors, gloo in the CPU tests."""
    if world_size == 1:
        full.copy_(local)
        return full
    import torch.distributed as dist
    dist.all_gather_into_tensor(full.view(-1), local.contiguous().view(-1), group=group)
    return full


class AdmmEngine:
    """All agents of a run, sharded over ranks in contiguous blocks (agent a lives on rank a // (A/world))."""

    def __init__(self, shards, theta0, psi0, *, rho, L, process_group=None, rank=0, world_size=1, streams=True, **agent_kw):
        _require_cuda()
        self._lib = _lib.load()
        self.A_total = int(theta0.shape[0])
        self.P = int(theta0.shape[1])
        self.world, self.rank, self.pg = int(world_size), int(rank), process_group
        block = agent_block(self.rank, self.world, self.A_total)
        self.A_local = len(block)
        if len(shards) != self.A_local:
            raise ValueError(f"rank {rank} expects {self.A_local} shards, got {len(shards)}")
        self.first = block.start
        self.rho = float(rho)
        lips = L if np.ndim(L) else [L] * self.A_total
        # one agent per GPU: latency matters -> rank-256 outer panels (measured best of 1, 2, 4, 6, 8 and of the 4-then-2
        # schedule, outer_blocks = -1, which ties with 2); several agents: throughput -> rank-512.  Shards up to 6144 samples are
        # bound by the leaf chain either way: the solver's size-aware default (rank-128 panels) is best for them.
        n_max = max(len(y) for _, y in shards)
        agent_kw.setdefault("cholesky_outer_blocks", 0 if n_max <= 6144 else (2 if self.A_local == 1 else 4))
        self.agents = [AgentEngine(x, y, rho=rho, L=lips[self.first + i], **agent_kw) for i, (x, y) in enumerate(shards)]
        if any(a.P != self.P for a in self.agents):
            raise ValueError("theta0 does not match the circuit's parameter count")
        # theta_a and psi_a side by side in ONE (A, 2, P) buffer: a single all-gather per iteration moves both
        self.rows = dev_f64(np.stack([np.asarray(theta0, dtype=np.float64), np.asarray(psi0, dtype=np.float64)], axis=1))
        self.theta, self.psi = self.rows[:, 0], self.rows[:, 1]              # (A, P) views, row stride 2P
        self.z = torch.empty(self.P, dtype=torch.float64, device=self.rows.device)
        self.local_rows = torch.empty((self.A_local, 2, self.P), dtype=torch.float64, device=self.rows.device)
        self.local_theta, self.local_psi = self.local_rows[:, 0], self.local_rows[:, 1]
        self._psi_before = torch.empty((self.A_local, self.P), dtype=torch.float64, device=self.rows.device)
        self.streams = [torch.cuda.Stream() for _ in self.agents] if (streams and self.A_local > 1) else None
        self.entries_per_iteration = sum(a.entries_per_step for a in self.agents)

    def consensus(self):
        check(self._lib.dqgp_admm_consensus_strided(self.theta.data_ptr(), self.psi.data_ptr(), self.A_total, self.P, 2 * self.P, self.rho,
                                                    PERIOD, self.z.data_ptr(), stream_ptr()), "consensus")

    def _local_part(self):
        """Consensus z (replicated, from the gathered theta/psi) and every local agent's step: device work only."""
        self.consensus()
        self._psi_before.copy_(self.psi[self.first:self.first + self.A_local])     # what repair_failed_agents restarts from
        if self.streams is None:
            for i, ag in enumerate(self.agents):
                ag.step(self.z, self.psi[self.first + i], self.local_theta[i], self.local_psi[i])
        else:
            main = torch.cuda.current_stream()
            ready = torch.cuda.Event()
            ready.record(main)
            for i, ag in enumerate(self.agents):
                s = self.streams[i]
                s.wait_event(ready)
                with torch.cuda.stream(s):
                    ag.step(self.z, self.psi[self.first + i], self.local_theta[i], self.local_psi[i])
                done = torch.cuda.Event()
                done.record(s)
                main.wait_event(done)

    def _exchange(self):
        exchange_rows(self.rows, self.local_rows, self.pg, self.world)      # ONE collective: (A_local, 2, P) -> (A, 2, P)

    def iteration(self):
        self._local_part()
        self._exchange()

    def repair_failed_agents(self):
        """Host check after an iteration (synchronises): every local agent whose Cholesky reported a non-positive pivot redoes
        its step down the reference's LU ladder (agent_riemannian.py:419-425) from the same z and psi, and the rows are
        exchanged again.  Returns the number of agents repaired on this rank (collective when world_size > 1: every rank
        must call it)."""
        infos = torch.stack([a.d_info[0] for a in self.agents]).cpu().numpy()
        bad = [i for i, v in enumerate(infos) if v != 0]
        for i in bad:
            # psi row of the agent as it was BEFORE this iteration's exchange overwrote it: kept in psi_before
            self.agents[i].step_fallback(self.z, self._psi_before[i], self.local_theta[i], self.local_psi[i])
        n_bad = torch.tensor([len(bad)], device=self.rows.device)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(n_bad, group=self.pg)
        if int(n_bad.item()) > 0:
            self._exchange()
        return len(bad)

    def capture(self):
        """Capture the device part of one iteration (consensus, all local agents, their streams and the solver's internal
        look-ahead streams) into a CUDA graph; `replay()` then costs one launch plus the row exchange, which stays
        outside the graph (an in-place copy on one rank, the NCCL all-gather on several).  The warm-up iteration that capture
        needs (lazy uploads, function attributes) does NOT advance the run: theta / psi / z are restored afterwards, so
        capture() + k replays walks exactly k iterations, like k eager iteration() calls."""
        keep = [t.clone() for t in (self.rows, self.z, self.local_rows)]
        self.iteration()                         # warm-up
        torch.cuda.synchronize()
        for t, k in zip((self.rows, self.z, self.local_rows), keep):
            t.copy_(k)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self._local_part()
        self._graph = graph
        return graph

    def replay(self):
        self._graph.replay()
        self._exchange()

    def hyper_gradients(self):
        """(A_local, k) array of the local agents' last hyper-gradients (synchronises; needs hyper_gradient=True): each row is
        [dNLL/dh in h_hyp order, dNLL/dsigma] (names in `agents[0].hyper_names` + "noise_std").  Every agent shares the
        hyper-parameters, so the sum over rows (and over ranks) is the gradient of the summed local NLLs."""
        if not all(a.hyper_gradient_enabled for a in self.agents):
            raise ValueError("hyper_gradients() needs AdmmEngine(..., hyper_gradient=True)")
        return torch.stack([a.d_hyper_grad for a in self.agents]).cpu().numpy()

    def state(self):
        """(z, theta, psi, per-agent NLL) on the host (synchronises)."""
        nll = np.array([float(a.d_nll[3].item()) for a in self.agents])
        return self.z.cpu().numpy(), self.theta.cpu().numpy(), self.psi.cpu().numpy(), nll
