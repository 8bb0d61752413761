"""GPU-backed quantum-kernel objects with the surface the reference uses on squlearn's
``FidelityKernel`` / ``ProjectedQuantumKernel`` (``main.py:43-145``; uses at ``main.py:199,205,245,1413,
1420-1430,2398-2400`` and ``agent_riemannian.py:114,118,379``): ``evaluate(x, y)``, ``assign_parameters(p)``,
writable ``_parameters``, ``num_parameters`` (``None`` before first use for the projected kernel),
``encoding_circuit.num_parameters`` and ``executor``.  All arithmetic runs in libdqgp (csrc/statevec.cu,
csrc/gram.cu); NumPy arrays cross the boundary, nothing is computed on the host.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import ENCODINGS, OUTER_KERNELS, DqgpError, check


def _require_cuda():
    if not torch.cuda.is_available():
        raise DqgpError("dqgp_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def dev_f64(a, device="cuda"):
    """Host array -> contiguous fp64 device tensor (through pinned memory so the copy is a real async H2D)."""
    t = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))
    return t.pin_memory().to(device, non_blocking=True) if t.numel() else t.to(device)


class EncodingCircuit:
    """Handle to a device-resident gate program (``dqgp_circuit``); named after squlearn's base class."""

    def __init__(self, encoding_type, num_qubits, num_features, num_layers):
        if encoding_type not in ENCODINGS:
            raise ValueError(f"Unknown encoding type: {encoding_type}. Supported on the hot path: {sorted(ENCODINGS)}")
        self.encoding_type = encoding_type
        self.num_qubits, self.num_features, self.num_layers = int(num_qubits), int(num_features), int(num_layers)
        self._lib = _lib.load()
        h = C.c_void_p()
        check(self._lib.dqgp_circuit_create(ENCODINGS[encoding_type], self.num_qubits, self.num_features,
                                            self.num_layers, C.byref(h)), "dqgp_circuit_create")
        self.handle = h
        self.num_parameters = self._lib.dqgp_circuit_num_parameters(h)
        self.num_gates = self._lib.dqgp_circuit_num_gates(h)

    def describe(self):
        buf = (_lib.Gate * self.num_gates)()
        check(self._lib.dqgp_circuit_describe(self.handle, buf, self.num_gates), "dqgp_circuit_describe")
        return [(g.kind, g.q0, g.q1, g.form, g.pidx, g.fidx, g.coef) for g in buf]

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self._lib.dqgp_circuit_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    # device-level helpers (tensors in, tensors out) -------------------------------------------------
    def features(self, d_x, d_pm):
        n, s = d_x.shape[0], d_pm.shape[0]
        out = torch.empty((s, n, 3 * self.num_qubits), dtype=torch.float64, device=d_x.device)
        check(self._lib.dqgp_features(self.handle, d_x.data_ptr(), n, d_pm.data_ptr(), s, out.data_ptr(), stream_ptr()),
              "dqgp_features")
        return out

    def states(self, d_x, d_pm):
        n, s = d_x.shape[0], d_pm.shape[0]
        out = torch.empty((s, n, 1 << self.num_qubits, 2), dtype=torch.float64, device=d_x.device)
        check(self._lib.dqgp_states(self.handle, d_x.data_ptr(), n, d_pm.data_ptr(), s, out.data_ptr(), stream_ptr()),
              "dqgp_states")
        return out


class Executor:
    """Name holder (both squlearn executors are exact shot-free simulators; the GPU path is too)."""

    def __init__(self, name="statevector_simulator"):
        self.name = name

    def __repr__(self):
        return f"Executor({self.name}) [dqgp_b200 statevector]"


def outer_hyp(outer_kernel, params=None):
    """Host hyper-parameter vector of an outer kernel: gaussian {gamma}; matern {length_scale} (nu = 1.5);
    expsinesquared {length_scale, periodicity}; rationalquadratic {length_scale, alpha}; dotproduct {sigma_0};
    pairwisekernel {0.0}: scikit-learn's PairwiseKernel(metric="linear") is f.g, the dot product with sigma_0 = 0 (its
    gamma is accepted and ignored, as filter_params=True does).  Defaults = the only values the reference reaches (Q2)."""
    params = dict(params or {})
    if outer_kernel == "gaussian":
        return [float(params.get("gamma", 1.0))]
    if outer_kernel == "matern":
        if float(params.get("nu", 1.5)) != 1.5:
            raise ValueError("only Matern nu=1.5 is on the hot path")
        return [float(params.get("length_scale", 1.0))]
    if outer_kernel == "expsinesquared":
        return [float(params.get("length_scale", 1.0)), float(params.get("periodicity", 1.0))]
    if outer_kernel == "rationalquadratic":
        return [float(params.get("length_scale", 1.0)), float(params.get("alpha", 1.0))]
    if outer_kernel == "dotproduct":
        return [float(params.get("sigma_0", 1.0))]
    if outer_kernel == "pairwisekernel":
        if params.get("metric", "linear") != "linear":
            raise ValueError(f"only PairwiseKernel metric='linear' is on the hot path (got {params['metric']!r})")
        return [0.0]
    raise ValueError(f"outer kernel {outer_kernel!r} is outside the hot path (supported: {sorted(OUTER_KERNELS)})")


class _QuantumKernel:
    def __init__(self, encoding_circuit, executor=None, parameter_seed=0):
        _require_cuda()
        self.encoding_circuit = encoding_circuit
        self.executor = executor if executor is not None else Executor()
        rng = np.random.default_rng(parameter_seed)
        self._parameters = rng.uniform(-np.pi, np.pi, encoding_circuit.num_parameters)
        self._lib = _lib.load()

    def assign_parameters(self, parameters):
        p = np.asarray(parameters, dtype=np.float64)
        if p.shape != (self.encoding_circuit.num_parameters,):
            raise ValueError(f"expected {self.encoding_circuit.num_parameters} parameters, got {p.shape}")
        self._parameters = p.copy()

    @property
    def parameters(self):
        return self._parameters

    def _inputs(self, x, y):
        d = self.encoding_circuit.num_features
        x = np.asarray(x, dtype=np.float64)
        x = x.reshape(-1, d) if x.ndim != 2 else x
        same = y is None or y is x
        y = x if same else np.asarray(y, dtype=np.float64)
        y = y.reshape(-1, d) if y.ndim != 2 else y
        if x.shape[1] != d or y.shape[1] != d:
            raise ValueError(f"expected {d} features per sample")
        d_x = dev_f64(x)
        d_y = d_x if same else dev_f64(y)
        d_p = dev_f64(np.asarray(self._parameters, dtype=np.float64).reshape(1, -1))
        return d_x, d_y, d_p, same


class FidelityKernel(_QuantumKernel):
    """K[j,k] = |<psi(y_k)|psi(x_j)>|^2 (reference main.py:118-124)."""

    def __init__(self, encoding_circuit, executor=None, parameter_seed=0, use_expectation=True,
                 evaluate_duplicates="all", **_ignored):
        super().__init__(encoding_circuit, executor, parameter_seed)
        self.num_parameters = encoding_circuit.num_parameters

    def evaluate(self, x, y=None):
        d_x, d_y, d_p, same = self._inputs(x, y)
        return self.evaluate_device(d_x, d_y, d_p, same).cpu().numpy()

    def evaluate_device(self, d_x, d_y, d_p, same=False, out=None, ld=None):
        enc = self.encoding_circuit
        s1 = enc.states(d_x, d_p)
        s2 = s1 if same else enc.states(d_y, d_p)
        n1, n2 = d_x.shape[0], d_y.shape[0]
        if out is None:
            out = torch.empty((n1, n2), dtype=torch.float64, device=d_x.device)
            ld = n2
        check(self._lib.dqgp_gram_fidelity(s1.data_ptr(), n1, s2.data_ptr(), n2, 1 << enc.num_qubits, out.data_ptr(), ld,
                                           int(same), stream_ptr()), "dqgp_gram_fidelity")
        return out


class ProjectedQuantumKernel(_QuantumKernel):
    """Outer kernel on the XYZ Pauli-expectation features (reference main.py:130-137)."""

    def __init__(self, encoding_circuit, measurement="XYZ", outer_kernel="gaussian", executor=None,
                 parameter_seed=0, regularization=None, **outer_kernel_params):
        super().__init__(encoding_circuit, executor, parameter_seed)
        if measurement != "XYZ":
            raise NotImplementedError("only measurement='XYZ' is on the hot path")
        if regularization is not None:
            raise NotImplementedError("regularization is outside the hot path (SURVEY §2 #13)")
        self.outer_kernel = str(outer_kernel).lower()
        self._hyp = outer_hyp(self.outer_kernel, outer_kernel_params)
        self.num_parameters = None      # squlearn quirk mirrored (main.py:198-199)

    def evaluate(self, x, y=None):
        d_x, d_y, d_p, same = self._inputs(x, y)
        self.num_parameters = self.encoding_circuit.num_parameters
        return self.evaluate_device(d_x, d_y, d_p, same).cpu().numpy()

    def evaluate_device(self, d_x, d_y, d_p, same=False, out=None, ld=None):
        enc = self.encoding_circuit
        f1 = enc.features(d_x, d_p)
        f2 = f1 if same else enc.features(d_y, d_p)
        n1, n2 = d_x.shape[0], d_y.shape[0]
        if out is None:
            out = torch.empty((n1, n2), dtype=torch.float64, device=d_x.device)
            ld = n2
        check(self._lib.dqgp_gram_projected(OUTER_KERNELS[self.outer_kernel], _lib.hyp_array(self._hyp), f1.data_ptr(), n1,
                                            f2.data_ptr(), n2, 3 * enc.num_qubits, out.data_ptr(), ld, int(same),
                                            stream_ptr()), "dqgp_gram_projected")
        return out


def create_quantum_kernel(num_qubits, num_features=1, num_layers=2, use_parameter_shift=True, encoding_type="yz_cx",
                          kernel_type="fidelity", measurement="XYZ", outer_kernel="gaussian", outer_kernel_params=None,
                          regularization=None):
    """Same signature and error behaviour as ``main.create_quantum_kernel`` (main.py:43-145).  As in the
    reference, ``outer_kernel_params`` are accepted and NOT applied (Q2): the outer kernel always runs with
    scikit-learn's defaults.  ``use_parameter_shift`` only picked the simulator backend there."""
    enc = EncodingCircuit(encoding_type, num_qubits, num_features, num_layers)
    executor = Executor("statevector_simulator" if use_parameter_shift else "pennylane")
    if kernel_type == "fidelity":
        return FidelityKernel(enc, executor=executor, parameter_seed=0)
    if kernel_type == "projected":
        return ProjectedQuantumKernel(enc, measurement=measurement, outer_kernel=outer_kernel, executor=executor,
                                      parameter_seed=0, regularization=regularization)
    raise ValueError(f"Unknown kernel type: {kernel_type}. Supported: 'fidelity', 'projected'")
