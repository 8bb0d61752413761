"""``RiemannianAgent`` and ``process_agent_training`` with the reference's constructor / call signatures
(``agent_riemannian.py:126-491``, ``main.py:1311-1362``), executing the whole step on the GPU.

Host arrays in, host arrays out: every call copies the agent's shard, z and psi_i to the device (the
reference pickles the same data to its worker processes every iteration) and reads back
``(theta_i, psi_i, nll_loss, condition_number, nll_components)``.  Both process pools of the reference
(agents x shifted-parameter jobs) collapse into one stream of kernels.

Reference behaviours kept: only the (2P+1)-evaluation central-difference path exists (Q3/Q4); training
Grams use the Gaussian outer kernel whatever ``outer_kernel`` says (Q1) unless
``training_ignores_outer_kernel=False``; gradient, theta_i and psi_i are rounded to 4 decimals (Q5);
``riemannian_*`` arguments are accepted and inert (Q8); a failed Cholesky walks the reference's LU rung on the device
(``agent_riemannian.py:419-425``).  Deviation, documented: ``condition_number`` is NaN
unless ``compute_condition_number=True`` (the reference's ``np.linalg.cond`` is an O(n^3) SVD used only in
prints, main.py:2629-2642).
"""
from __future__ import annotations

import numpy as np
import torch

from .engine import AgentEngine
from .kernels import dev_f64
from .riemannian import create_riemannian_framework

_ENGINE_CACHE = {}     # per-process, like the reference's per-process kernel cache (main.py:147-159)


def _engine_for(key, factory):
    eng = _ENGINE_CACHE.get(key)
    if eng is None:
        if len(_ENGINE_CACHE) >= 64:
            _ENGINE_CACHE.clear()
        eng = _ENGINE_CACHE[key] = factory()
    return eng


class RiemannianAgent:
    def __init__(self, agent_id, X_sub, Y_sub, num_qubits, noise_std, rho, L, q_kernel=None, use_parameter_shift=False,
                 num_workers=None, shift_value=np.pi / 8, num_layers=2, combined_computation=True, encoding_type="yz_cx",
                 kernel_type="fidelity", measurement="XYZ", outer_kernel="gaussian", outer_kernel_params=None,
                 regularization=None, riemannian_lr=0.01, riemannian_method="gradient_descent", riemannian_beta=0.9,
                 training_ignores_outer_kernel=None, compute_condition_number=False, gradient=None, reupload_shard="if_changed"):
        # use_parameter_shift selects the reference's branch (agent_riemannian.py:383-404):
        #   True  (what main.py hard-codes, :2301): the (2P+1)-job workers, whose config dict carries no outer kernel -> Gaussian
        #         training Grams (Q1), central difference with h = shift_value;
        #   False, projected: `_manual_projected_kernel_derivatives_riemannian` (:279-312) - the same central difference, but
        #         through self.q_kernel, which was built with the REAL outer kernel -> training_ignores_outer_kernel=False;
        #   False, fidelity: `q_kernel.evaluate_derivatives(["K", "dKdp"])` (:402-404), the analytic derivative -> gradient="analytic"
        #         (every qubit count up to 12, as the central difference).
        # Explicit `training_ignores_outer_kernel` / `gradient` arguments override the mapping.
        if training_ignores_outer_kernel is None:
            training_ignores_outer_kernel = bool(use_parameter_shift) or kernel_type != "projected"
        if gradient is None:
            gradient = "analytic" if (not use_parameter_shift and kernel_type == "fidelity") else "central_difference"
        self.gradient = gradient
        # "if_changed": X_sub / Y_sub stay resident on the GPU and are re-uploaded only when they differ from the staged copy;
        # "always": copy them every call, as the reference re-pickles them to its workers every iteration (main.py:2530-2542)
        self.reupload_shard = reupload_shard
        import os
        self.use_cuda_graph = os.environ.get("DQGP_AGENT_GRAPH", "1") != "0"
        self.agent_id = agent_id
        self.X_sub = np.asarray(X_sub, dtype=np.float64)
        if self.X_sub.ndim == 1:
            self.X_sub = self.X_sub.reshape(-1, 1)
        self.Y_sub = np.asarray(Y_sub, dtype=np.float64).reshape(-1)
        self.num_qubits, self.noise_std, self.rho, self.L = num_qubits, noise_std, rho, L
        self.q_kernel, self.use_parameter_shift, self.num_workers = q_kernel, use_parameter_shift, num_workers
        self.shift_value, self.num_layers, self.combined_computation = shift_value, num_layers, combined_computation
        self.encoding_type, self.kernel_type, self.measurement = encoding_type, kernel_type, measurement
        self.outer_kernel, self.outer_kernel_params, self.regularization = outer_kernel, outer_kernel_params, regularization
        self.riemannian_lr, self.riemannian_method, self.riemannian_beta = riemannian_lr, riemannian_method, riemannian_beta
        self.training_ignores_outer_kernel = training_ignores_outer_kernel
        self.compute_condition_number = compute_condition_number
        self.manifold = self.riemannian_optimizer = self.riemannian_admm = None
        if measurement != "XYZ":
            raise NotImplementedError("only measurement='XYZ' is on the hot path")
        if regularization is not None:
            raise NotImplementedError("regularization is outside the hot path (SURVEY §2 #13)")
        self.last_gradient = None       # unrounded dL/dtheta of the last call (diagnostics / tests)
        self.h2d_bytes = self.d2h_bytes = 0

    def _setup_riemannian_framework(self, num_parameters):
        if self.manifold is None:
            self.manifold, self.riemannian_optimizer, self.riemannian_admm = create_riemannian_framework(
                num_parameters=num_parameters, learning_rate=self.riemannian_lr, rho=self.rho, method=self.riemannian_method)

    def _engine(self):
        n, d = self.X_sub.shape
        key = (self.agent_id, n, d, self.encoding_type, self.kernel_type, self.num_qubits, self.num_layers, self.outer_kernel,
               float(self.noise_std), float(self.rho), float(self.L), float(self.shift_value), self.training_ignores_outer_kernel,
               self.gradient)
        return _engine_for(key, lambda: AgentEngine(
            self.X_sub, self.Y_sub, encoding_type=self.encoding_type, kernel_type=self.kernel_type, num_qubits=self.num_qubits,
            num_layers=self.num_layers, noise_std=self.noise_std, rho=self.rho, L=self.L, outer_kernel=self.outer_kernel,
            shift_value=self.shift_value, training_ignores_outer_kernel=self.training_ignores_outer_kernel, gradient=self.gradient))

    def train_and_update(self, z, psi_i):
        """-> (theta_i, psi_i, nll_loss, condition_number, nll_components), as agent_riemannian.py:491."""
        return self.collect(self.submit(z, psi_i))

    def submit(self, z, psi_i, stream=None):
        """Enqueue the whole step (H2D of shard, z, psi; all kernels; packing of the result) on `stream` without
        waiting for it.  `collect()` reads the result back.  Lets a driver overlap the agents of one GPU — the
        reference overlaps them with a process pool (main.py:2530-2542)."""
        eng = self._engine()
        z = np.asarray(z, dtype=np.float64).reshape(-1)
        psi_i = np.asarray(psi_i, dtype=np.float64).reshape(-1)
        if z.size != eng.P or psi_i.size != eng.P:
            raise ValueError(f"expected {eng.P} parameters, got z {z.size}, psi {psi_i.size}")
        self._setup_riemannian_framework(eng.P)
        ctx = torch.cuda.stream(stream) if stream is not None else _NullCtx()
        if getattr(eng, "_d_in", None) is None:
            eng._d_in = torch.empty((2, eng.P), dtype=torch.float64, device=eng.d_X.device)
            eng._d_out = torch.empty((3 * eng.P + 5,), dtype=torch.float64, device=eng.d_X.device)
            eng._graph, eng._graph_busy, eng._eager_calls = None, False, 0
        d_in, d_out, p = eng._d_in, eng._d_out, eng.P

        def enqueue(h_in, h_out):
            """H2D of z / psi, the whole step, packing of the result, one D2H: ~100 launches, or one CUDA-graph launch."""
            d_in.copy_(h_in, non_blocking=True)
            eng.step(d_in[0], d_in[1], d_out[:p], d_out[p:2 * p])
            d_out[2 * p:2 * p + 4].copy_(eng.d_nll)
            d_out[2 * p + 4:3 * p + 4].copy_(eng.d_grad)
            d_out[3 * p + 4:].copy_(eng.d_info)                 # int32 -> float64
            h_out.copy_(d_out, non_blocking=True)

        # From the second call on, the step replays as ONE CUDA graph (the engine's own pinned staging pair is baked into its
        # copy nodes); a call that arrives while that pair is still in flight, or DQGP_AGENT_GRAPH=0, takes the eager path.
        use_graph = self.use_cuda_graph and not eng._graph_busy and eng._eager_calls >= 1
        if use_graph and eng._graph is None:
            eng._g_pair = eng.staging()
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                enqueue(*eng._g_pair)
            eng._graph = graph
        pair = eng._g_pair if use_graph else eng.staging()      # persistent pinned buffers (no cudaHostAlloc per call)
        h_in, h_out = pair
        h_in[0].copy_(torch.from_numpy(z))
        h_in[1].copy_(torch.from_numpy(psi_i))
        with ctx:
            shard_bytes = eng.load_data(self.X_sub, self.Y_sub, always=self.reupload_shard == "always")
            if use_graph:
                eng._graph.replay()
                eng._graph_busy = True
            else:
                enqueue(h_in, h_out)
                eng._eager_calls += 1
            done = torch.cuda.Event()
            done.record()
        self.h2d_bytes = shard_bytes + z.nbytes + psi_i.nbytes
        self.d2h_bytes = h_out.numel() * 8
        return (eng, d_in, (pair, use_graph), h_out, done)

    def collect(self, pending):
        eng, d_in, (pair, used_graph), host, done = pending
        done.synchronize()
        packed = host.numpy().copy()
        if used_graph:
            eng._graph_busy = False
        else:
            eng.release(pair)
        p = eng.P
        theta_i, psi_new = packed[:p].copy(), packed[p:2 * p].copy()
        terms = packed[2 * p:2 * p + 4]
        self.last_gradient = packed[2 * p + 4:3 * p + 4].copy()
        info = int(packed[-1])
        if info != 0:
            # np.linalg.cholesky raised in the reference: its except-branch refactors with LU (agent_riemannian.py:419-425).
            # Same here, on the device: full symmetric Gram, partial-pivoting LU, alpha / explicit inverse / slogdet.
            d_out = eng._d_out
            eng.step_fallback(d_in[0], d_in[1], d_out[:p], d_out[p:2 * p])
            d_out[2 * p:2 * p + 4].copy_(eng.d_nll)
            d_out[2 * p + 4:3 * p + 4].copy_(eng.d_grad)
            packed = d_out.cpu().numpy()
            theta_i, psi_new = packed[:p].copy(), packed[p:2 * p].copy()
            terms = packed[2 * p:2 * p + 4]
            self.last_gradient = packed[2 * p + 4:3 * p + 4].copy()
            self.used_lu_fallback = True
        cond = float("nan")
        if self.compute_condition_number:
            eng.simulate(d_in[0]); eng.gram()      # the solver matrix holds L after the step: rebuild K for the diagnostic
            k = torch.tril(eng.solver.matrix()); k = k + k.T - torch.diag(torch.diagonal(k))
            k = k - (self.noise_std ** 2) * torch.eye(eng.n, dtype=torch.float64, device=k.device)
            sv = torch.linalg.svdvals(k)
            cond = float((sv[0] / sv[-1]).item())
        comps = {"log_det_term": float(terms[0]), "quadratic_term": float(terms[1]), "constant_term": float(terms[2]),
                 "total": float(terms[3])}
        return theta_i, psi_new, float(terms[3]), cond, comps


class _NullCtx:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def train_agents(agents, z, psis, streams=None):
    """Run `train_and_update(z, psis[i])` for several agents of this GPU concurrently (one CUDA stream each) and
    return the list of 5-tuples in agent order — the GPU counterpart of the reference's
    `executor.map(process_agent_training, ...)` fan-out (main.py:2530-2542).  Agents must have distinct shard shapes
    or configurations only if they are meant to share nothing: engines are cached per (shape, configuration), so
    agents with identical keys are serialised on one engine."""
    if streams is None:
        streams = [torch.cuda.Stream() for _ in agents]
    main = torch.cuda.current_stream()
    ready = torch.cuda.Event()
    ready.record(main)
    pending, seen = [], {}
    for ag, psi, st in zip(agents, psis, streams):
        key = id(ag._engine())
        if key in seen:                       # same cached engine: keep program order on its stream
            st = seen[key]
        seen[key] = st
        st.wait_event(ready)
        pending.append(ag.submit(z, psi, stream=st))
    return [ag.collect(p) for ag, p in zip(agents, pending)]


def process_agent_training(agent_data):
    """Same 23-tuple in / 5-tuple out as ``main.process_agent_training`` (main.py:1311-1362)."""
    (agent_id, X_sub, Y_sub, num_qubits, noise_std, rho, L, z, psi_i, use_parameter_shift, num_features, num_layers,
     num_workers, shift_value, encoding_type, kernel_type, measurement, riemannian_lr, riemannian_method, riemannian_beta,
     outer_kernel, outer_kernel_params, regularization) = agent_data
    agent = RiemannianAgent(agent_id=agent_id, X_sub=X_sub, Y_sub=Y_sub, num_qubits=num_qubits, noise_std=noise_std, rho=rho,
                            L=L, q_kernel=None, use_parameter_shift=use_parameter_shift, num_workers=num_workers,
                            shift_value=shift_value, num_layers=num_layers, encoding_type=encoding_type,
                            kernel_type=kernel_type, measurement=measurement, outer_kernel=outer_kernel,
                            outer_kernel_params=outer_kernel_params, regularization=regularization,
                            riemannian_lr=riemannian_lr, riemannian_method=riemannian_method, riemannian_beta=riemannian_beta)
    return agent.train_and_update(z, psi_i)
