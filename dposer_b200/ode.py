"""Explicit Runge-Kutta 4(5) (Dormand-Prince) with scipy's step-size controller on the host and all vector arithmetic in
native kernels -- the device-side replacement of ``scipy.integrate.solve_ivp(..., method='RK45')`` as the reference
drives it (lib/algorithms/advanced/likelihood.py:93-101, sampling.py:520-524).

The controller below restates scipy 1.x ``RungeKutta._step_impl`` / ``select_initial_step`` (SAFETY 0.9, factors in
[0.2, 10], error exponent -1/5, RMS error norm over the whole state vector); the arithmetic it drives is abstract
(:class:`Backend`), so the CPU test runs the same controller over a numpy backend against ``solve_ivp`` itself, and the
product path runs it over :class:`PFOdeBackend` (state in fp64 on the GPU; one scalar read back per attempted step).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L
from . import utils as mutils

SAFETY, MIN_FACTOR, MAX_FACTOR = 0.9, 0.2, 10.0
C_NODES = (0.0, 1 / 5, 3 / 10, 4 / 5, 8 / 9, 1.0)
ERROR_EXPONENT = -1.0 / 5.0


class Backend:
    """What the controller needs.  k[0..6] are the stage derivatives, y the accepted state, y_new the candidate."""
    n = 0

    def eval_initial(self, t):            # k[0] = f(t, y)
        raise NotImplementedError

    def eval_stage(self, s, t, h):        # k[s] = f(t, y + h sum_j a[s][j] k_j),  s = 1..5
        raise NotImplementedError

    def eval_candidate(self, t, h):       # y_new = y + h sum_j b_j k_j ; k[6] = f(t, y_new)
        raise NotImplementedError

    def error_norm(self, h, rtol, atol):  # rms(h sum_j e_j k_j / (atol + rtol max(|y|, |y_new|)))
        raise NotImplementedError

    def accept(self):                     # y <- y_new ; k[0] <- k[6]
        raise NotImplementedError

    def initial_step_norms(self, t0, direction, rtol, atol, interval):   # -> h_abs (select_initial_step)
        raise NotImplementedError


def select_initial_step(y0, f0, eval_f, t0, direction, rtol, atol, interval, order=4):
    """scipy.integrate._ivp.common.select_initial_step on host vectors (a one-time cost: three vector copies)."""
    if interval == 0.0:
        return 0.0
    rms = lambda v: np.linalg.norm(v) / v.size ** 0.5      # noqa: E731
    scale = atol + np.abs(y0) * rtol
    d0, d1 = rms(y0 / scale), rms(f0 / scale)
    h0 = 1e-6 if (d0 < 1e-5 or d1 < 1e-5) else 0.01 * d0 / d1
    h0 = min(h0, interval)
    f1 = eval_f(t0 + h0 * direction, y0 + h0 * direction * f0)
    d2 = rms((f1 - f0) / scale) / h0
    if d1 <= 1e-15 and d2 <= 1e-15:
        h1 = max(1e-6, h0 * 1e-3)
    else:
        h1 = (0.01 / max(d1, d2)) ** (1 / (order + 1))
    return min(100 * h0, h1, interval)


def solve_rk45(backend, t0, t_bound, rtol=1e-3, atol=1e-6, max_attempts=1000000):
    """Integrate from t0 to t_bound; the final state is ``backend``'s accepted y.  Returns (nfev, attempted steps)."""
    rtol = max(rtol, 100 * np.finfo(float).eps)            # scipy's validate_tol
    direction = float(np.sign(t_bound - t0)) if t_bound != t0 else 1.0
    backend.eval_initial(t0)
    nfev = 1
    h_abs = backend.initial_step_norms(t0, direction, rtol, atol, abs(t_bound - t0))
    nfev += 1
    t, attempts = float(t0), 0
    while direction * (t - t_bound) < 0:
        min_step = 10 * abs(np.nextafter(t, direction * np.inf) - t)
        h_abs = max(h_abs, min_step)
        step_rejected = False
        while True:
            attempts += 1
            if h_abs < min_step or attempts > max_attempts:
                raise RuntimeError('RK45: required step size is less than spacing between numbers')
            h = h_abs * direction
            t_new = t + h
            if direction * (t_new - t_bound) > 0:
                t_new = t_bound
            h = t_new - t
            h_abs = abs(h)
            for s in range(1, 6):
                backend.eval_stage(s, t + C_NODES[s] * h, h)
            backend.eval_candidate(t + h, h)
            nfev += 6
            err = backend.error_norm(h, rtol, atol)
            if err < 1:
                factor = MAX_FACTOR if err == 0 else min(MAX_FACTOR, SAFETY * err ** ERROR_EXPONENT)
                if step_rejected:
                    factor = min(1.0, factor)
                h_abs *= factor
                break
            h_abs *= max(MIN_FACTOR, SAFETY * err ** ERROR_EXPONENT)
            step_rejected = True
        backend.accept()
        t = t_new
    return nfev, attempts


class PFOdeBackend(Backend):
    """Probability-flow ODE of the score model on the GPU: state [x (B*D) | logp (B)] (``with_div``) or x alone, in fp64,
    with D the network's width (63 or 126); a function evaluation is the score net (+ its JVP along ``epsilon``) and
    ``dpb_pf_ode_rhs_dim``."""

    def __init__(self, model, sde, x0, epsilon=None):
        model.check_width(x0, 'x')
        if epsilon is not None:
            model.check_width(epsilon, 'epsilon', x0.shape[0])
        L.require_cuda(x0, 'x')
        self.model, self.sde, self.dev = model, sde, x0.device
        self.B, self.D = x0.shape[0], int(model.pose_width)
        self.nx = self.B * self.D
        self.with_div = epsilon is not None
        self.n = self.nx + (self.B if self.with_div else 0)
        self.eps = None if epsilon is None else epsilon.to(device=self.dev, dtype=torch.float32).contiguous()
        self.y = torch.zeros(self.n, dtype=torch.float64, device=self.dev)
        self.y[:self.nx] = x0.reshape(-1).double()
        self.y_new = torch.zeros_like(self.y)
        self.k = torch.zeros(7, self.n, dtype=torch.float32, device=self.dev)
        self.xs = torch.empty(self.B, self.D, dtype=torch.float32, device=self.dev)
        self.score = torch.empty_like(self.xs)
        self.jv = torch.empty_like(self.xs)
        self.lib = L.load()
        self.h = model.handle()
        self.scratch = torch.empty(int(self.lib.dpb_rk45_scratch_bytes()), dtype=torch.uint8, device=self.dev)
        nws = int(self.lib.dpb_score_jvp_workspace_bytes(self.h.ptr, self.B)) if self.with_div else 0
        self.ws = torch.empty(nws, dtype=torch.uint8, device=self.dev) if nws else None

    # ---- one function evaluation: xs (fp32 [B,D]) at time t -> k[i]
    def _f(self, t, i):
        tt = torch.tensor([float(t)], dtype=torch.float32)
        coef, label = mutils.em_coefficients(self.sde, self.model, tt, probability_flow=True, continuous=True)
        m = float(coef[0, 5])
        fx, g = self.sde.sde(torch.ones(1, 1), tt)
        fx, g2 = float(fx[0, 0]), float(g[0] ** 2)
        st = L.current_stream(self.dev)
        if self.with_div:
            table = self.model.time_table(label)
            L.check(self.lib.dpb_score_jvp(self.h.ptr, L.ptr(self.xs), L.ptr(self.eps), L.ptr(table[0]), None, None, m,
                                           L.ptr(self.score), L.ptr(self.jv), self.B, L.ptr(self.ws), self.ws.numel(), st))
            L.check(self.lib.dpb_pf_ode_rhs_dim(L.ptr(self.xs), L.ptr(self.score), L.ptr(self.jv), L.ptr(self.eps), fx, g2,
                                                L.ptr(self.k[i]), self.B, self.D, st))
        else:
            score = self.model.raw_forward(self.xs, label, torch.tensor([m]))
            L.check(self.lib.dpb_pf_ode_rhs_dim(L.ptr(self.xs), L.ptr(score), None, None, fx, g2, L.ptr(self.k[i]), self.B,
                                                self.D, st))

    def _stage(self, s, h, y_out):
        L.check(self.lib.dpb_rk45_stage(L.ptr(self.y), L.ptr(self.k), self.n, float(h), s, L.ptr(y_out), L.ptr(self.xs),
                                        self.nx, L.current_stream(self.dev)))

    def eval_initial(self, t):
        self.xs.copy_(self.y[:self.nx].view(self.B, -1))
        self._f(t, 0)

    def eval_stage(self, s, t, h):
        self._stage(s, h, None)
        self._f(t, s)

    def eval_candidate(self, t, h):
        self._stage(6, h, self.y_new)
        self._f(t, 6)

    def error_norm(self, h, rtol, atol):
        L.check(self.lib.dpb_rk45_error(L.ptr(self.y), L.ptr(self.y_new), L.ptr(self.k), self.n, float(h), float(rtol),
                                        float(atol), L.ptr(self.scratch), L.current_stream(self.dev)))
        return float(np.sqrt(float(self.scratch[:8].view(torch.float64)[0]) / self.n))      # the one read-back per step

    def accept(self):
        self.y, self.y_new = self.y_new, self.y
        self.k[0].copy_(self.k[6])

    def initial_step_norms(self, t0, direction, rtol, atol, interval):
        y0, f0 = self.y.cpu().numpy(), self.k[0].double().cpu().numpy()

        def eval_f(t, y1):
            self.xs.copy_(torch.from_numpy(y1[:self.nx]).to(self.dev).float().view(self.B, -1))
            self._f(t, 1)
            return self.k[1].double().cpu().numpy()
        return select_initial_step(y0, f0, eval_f, t0, direction, rtol, atol, interval)
