"""Log-likelihood / latent code under the probability-flow ODE with the reference's call surface
(lib/algorithms/advanced/likelihood.py:40-113).

``get_likelihood_fn(sde, inverse_scaler, ...)`` returns ``likelihood_fn(model, data) -> (bpd, z, nfe)``.  ``method='RK45'``
(the reference's) integrates on the device (ode.py: scipy's controller, native stage / error kernels); other methods fall
back to scipy on the host over the same function evaluation.  Every function evaluation is ONE native call,
``dpb_score_jvp``: the score net and its forward-mode derivative along the Hutchinson probe (split-fp16 tcgen05 GEMMs).  The
reference gets ``eps . (J^T eps)`` from autograd (likelihood.py:26-37); the same scalar is ``eps . (J eps)``, so no
backward pass through the network is needed.  drift and divergence follow from the affine form of the reverse SDE:

    drift = f_x x - 0.5 g^2 score,   score = -raw / (sigma std)      div = f_x sum(eps^2) + 0.5 g^2 / (sigma std) eps.(J_raw eps)
"""
import numpy as np
import torch
from scipy import integrate

from . import _lib as L
from . import utils as mutils


def drift_and_div(model, sde, x, t, epsilon, ws=None):
    """(drift [B,63], div [B]) of the probability-flow ODE at the batch-uniform time ``t`` (python float)."""
    L.require_cuda(x, 'x')
    B = x.shape[0]
    tt = torch.tensor([float(t)], dtype=torch.float32)
    # score = m * raw and the time label, evaluated by the same helper that builds the samplers' step tables
    # (VP / subVP: m = -1 / (sigma std), label = 999 t;  VE: m = +1 / sigma, label = sigma(t))
    coef, label = mutils.em_coefficients(sde, model, tt, probability_flow=True, continuous=True)
    m = float(coef[0, 5])
    fx, g = sde.sde(torch.ones(1, 1), tt)                  # f(x,t) = fx * x   (host fp32, like the reference's scalars)
    fx, g2 = float(fx[0, 0]), float(g[0] ** 2)
    table = model.time_table(label)
    h = model.handle()
    if ws is None:
        ws = torch.empty(int(L.load().dpb_score_jvp_workspace_bytes(h.ptr, B)), dtype=torch.uint8, device=x.device)
    score = torch.empty_like(x)
    jv = torch.empty_like(x)
    xc, ec = x.contiguous(), epsilon.contiguous()
    L.check(L.load().dpb_score_jvp(h.ptr, L.ptr(xc), L.ptr(ec), L.ptr(table[0]), None, None, m,
                                   L.ptr(score), L.ptr(jv), B, L.ptr(ws), ws.numel(), L.current_stream(x.device)))
    drift = fx * xc - 0.5 * g2 * score
    div = fx * (ec * ec).sum(dim=1) - 0.5 * g2 * (jv * ec).sum(dim=1)
    return drift, div


def get_likelihood_fn(sde, inverse_scaler, hutchinson_type='Rademacher', rtol=1e-5, atol=1e-5, method='RK45', eps=1e-5):
    """likelihood.py:40-113.  ``likelihood_fn(model, data, epsilon=None)``: ``epsilon`` fixes the probe (parity tests)."""

    def likelihood_fn(model, data, epsilon=None):
        if getattr(model, 'is_rot6d', False):
            raise NotImplementedError('likelihood evaluation (score-network JVP) is built for the 63-D axis network, not '
                                      'for rot6d (126-D) score networks')
        with torch.no_grad():
            L.require_cuda(data, 'data')
            data = data.to(torch.float32)
            shape = data.shape
            if epsilon is None:
                if hutchinson_type == 'Gaussian':
                    epsilon = torch.randn_like(data)
                elif hutchinson_type == 'Rademacher':
                    epsilon = torch.randint_like(data, low=0, high=2).float() * 2 - 1.
                else:
                    raise NotImplementedError(f"Hutchinson type {hutchinson_type} unknown.")
            epsilon = epsilon.to(device=data.device, dtype=torch.float32)
            if method == 'RK45':
                # device-side Dormand-Prince (ode.py): state [x | logp] in fp64 on the GPU, scipy's controller on the host,
                # one scalar read back per attempted step
                from . import ode
                be = ode.PFOdeBackend(model, sde, data, epsilon)
                nfe, _ = ode.solve_rk45(be, eps, sde.T, rtol=rtol, atol=atol)
                z = be.y[:be.nx].view(shape).to(torch.float32)
                delta_logp = be.y[be.nx:].to(torch.float32)
            else:
                h = model.handle()
                ws = torch.empty(int(L.load().dpb_score_jvp_workspace_bytes(h.ptr, shape[0])), dtype=torch.uint8,
                                 device=data.device)

                def ode_func(t, x):
                    sample = mutils.from_flattened_numpy(x[:-shape[0]], shape).to(data.device).type(torch.float32)
                    drift, div = drift_and_div(model, sde, sample, t, epsilon, ws)
                    return np.concatenate([mutils.to_flattened_numpy(drift), mutils.to_flattened_numpy(div)], axis=0)

                init = np.concatenate([mutils.to_flattened_numpy(data), np.zeros((shape[0],))], axis=0)
                solution = integrate.solve_ivp(ode_func, (eps, sde.T), init, rtol=rtol, atol=atol, method=method)
                nfe = solution.nfev
                zp = solution.y[:, -1]
                z = mutils.from_flattened_numpy(zp[:-shape[0]], shape).to(data.device).type(torch.float32)
                delta_logp = mutils.from_flattened_numpy(zp[-shape[0]:], (shape[0],)).to(data.device).type(torch.float32)
            prior_logp = sde.prior_logp(z)
            bpd = -(prior_logp + delta_logp) / np.log(2)
            bpd = bpd / np.prod(shape[1:])
            return bpd, z, nfe

    return likelihood_fn
