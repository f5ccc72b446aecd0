"""score_fn / model_fn wrappers (reference lib/algorithms/advanced/utils.py:95-186) and the
host-side scalar tables the fused kernels consume.

All scalar schedules are evaluated with the reference's own fp32 torch expressions on the CPU
(never in fp64, never in-kernel) so integer indices (``labels.long()``) and coefficients match
the reference bit for bit; only the resulting small tables are uploaded.
"""
import numpy as np
import torch

from . import _lib as L
from . import sde_lib


def get_model_fn(model, train=False):
    """utils.py:95-124."""
    def model_fn(x, labels, condition, mask):
        if train:
            raise NotImplementedError('training mode is out of scope for dposer_b200')
        model.eval()
        return model(x, labels, condition, mask)
    return model_fn


def _is_vp(sde):
    return isinstance(sde, (sde_lib.VPSDE, sde_lib.subVPSDE))


def get_score_fn(sde, model, train=False, continuous=False):
    """utils.py:127-186: labels = t*999, score = -model(x, labels)/std(t) (VP / subVP);
    VE: labels = sigma(t), score = model(x, labels)."""
    if train:
        raise NotImplementedError('training mode is out of scope for dposer_b200')
    if _is_vp(sde):
        def score_fn(x, t, condition=None, mask=None):
            model.eval()
            t = t.detach().to('cpu', torch.float32)       # schedule scalars are evaluated on the host (fp32)
            if continuous or isinstance(sde, sde_lib.subVPSDE):
                labels = t * 999
                std = sde.marginal_prob(torch.zeros_like(t)[:, None], t)[1]
            else:
                labels = t * (sde.N - 1)
                std = sde.sqrt_1m_alphas_cumprod[labels.long()]
            mult = -1.0 / std
            if model.config.model.scale_by_sigma:
                mult = mult / model._sigmas_host()[labels.long()]
            return model.raw_forward(x, labels, mult)
    elif isinstance(sde, sde_lib.VESDE):
        def score_fn(x, t, condition=None, mask=None):
            model.eval()
            if continuous:
                labels = sde.marginal_prob(torch.zeros_like(t)[:, None], t)[1]
            else:
                labels = torch.round((sde.T - t) * (sde.N - 1)).long()
            return model(x, labels, condition, mask)
    else:
        raise NotImplementedError(f"SDE class {sde.__class__.__name__} not yet supported.")
    return score_fn


def to_flattened_numpy(x):
    return x.detach().cpu().numpy().reshape((-1,))


def from_flattened_numpy(x, shape):
    return torch.from_numpy(x.reshape(shape))


# ---------------------------------------------------------------------------------------------
# scalar tables for the fused kernels
# ---------------------------------------------------------------------------------------------
def timestep_grid(sde, eps):
    """sampling.py:449 / run/completion.py:177: linspace(T, eps, N) in fp32 (CPU)."""
    return torch.linspace(sde.T, eps, sde.N)


def sigma_at(model, labels):
    """sigmas[floor(label)] (model.py:159) on the CPU copy of the buffer; 1 if scale_by_sigma is off."""
    if not model.config.model.scale_by_sigma:
        return torch.ones_like(labels)
    return model._sigmas_host()[labels.long()]


def em_coefficients(sde, model, t, probability_flow=False, continuous=True, predictor='euler_maruyama'):
    """Per-step affine form of a predictor for a CPU fp32 vector of times ``t``:

        x_mean = a x + b raw ,  x = x_mean + c z ,  impute with alpha/std

    where raw is the post_dense output before the sigma division (score = -raw / (sigma * std)).
      euler_maruyama      sampling.py:182-188 with sde_lib.py:98-106 and utils.py:152-162
      reverse_diffusion   sampling.py:210-220 with RSDE.discretize sde_lib.py:108-114 (f, G from SDE.discretize :52-69, or
                          VPSDE's DDPM rule :129-134); the reference's probability-flow factor there is 1.0, not 0.5
      ancestral_sampling  sampling.py:223-259, VPSDE (x + beta score) / sqrt(1 - beta) + sqrt(beta) z, VESDE the SMLD rule
    VESDE (sde_lib.py:234-295) takes the same three forms with score = +raw / sigma and labels = sigma(t).
    Returns (coef [n,8], labels [n]).
    """
    if predictor not in ('euler_maruyama', 'reverse_diffusion', 'ancestral_sampling'):
        raise NotImplementedError(f'predictor {predictor!r} is not supported')
    ve = isinstance(sde, sde_lib.VESDE)
    if not (_is_vp(sde) or ve):
        raise NotImplementedError(f'SDE class {sde.__class__.__name__} not yet supported.')
    t = t.to(torch.float32).cpu()
    one = torch.ones(t.numel(), 1)
    fx, g = sde.sde(one, t)                     # drift for x = 1  ->  f(x,t) = fx * x  (0 for VE)
    fx = fx[:, 0]
    # m: score = m * raw, raw = post_dense output before the sigma division (utils.py:127-180)
    if ve:
        labels = sde.marginal_prob(one, t)[1] if continuous else torch.round((sde.T - t) * (sde.N - 1))
        m = 1.0 / sigma_at(model, labels)
    else:
        if continuous or isinstance(sde, sde_lib.subVPSDE):
            labels = t * 999
            std_score = sde.marginal_prob(torch.zeros(t.numel(), 1), t)[1]
        else:
            labels = t * (sde.N - 1)
            std_score = sde.sqrt_1m_alphas_cumprod[labels.long()]
        m = -1.0 / (sigma_at(model, labels) * std_score)
    if predictor == 'euler_maruyama':
        dt = -1. / sde.N
        w = 0.5 if probability_flow else 1.0
        a = 1.0 + fx * dt
        b = -(g ** 2) * w * dt * m                   # x + (f - g^2 w score) dt
        c = torch.zeros_like(g) if probability_flow else g * float(np.sqrt(-dt))
    elif predictor == 'reverse_diffusion':
        ts = (t * (sde.N - 1) / sde.T).long()
        if isinstance(sde, sde_lib.VPSDE):           # DDPM discretisation: f = (sqrt(alpha) - 1) x, G = sqrt(beta)
            fd, G = torch.sqrt(sde.alphas[ts]) - 1.0, torch.sqrt(sde.discrete_betas[ts])
        elif ve:                                     # SMLD discretisation (sde_lib.py:277-285): f = 0, G^2 = sigma_i^2 - sigma_{i-1}^2
            sg = sde.discrete_sigmas[ts]
            adj = torch.where(ts == 0, torch.zeros_like(sg), sde.discrete_sigmas[ts - 1])
            fd, G = torch.zeros_like(sg), torch.sqrt(sg ** 2 - adj ** 2)
        else:                                        # f = drift / N, G = diffusion * sqrt(1 / N)
            fd, G = fx * (1. / sde.N), g * torch.sqrt(torch.tensor(1. / sde.N))
        a = 1.0 - fd                                 # x_mean = x - (f - G^2 score)
        b = (G ** 2) * m
        c = torch.zeros_like(G) if probability_flow else G
    else:
        if not isinstance(sde, (sde_lib.VPSDE, sde_lib.VESDE)):
            raise NotImplementedError(f'SDE class {sde.__class__.__name__} not yet supported.')
        assert not probability_flow, 'Probability flow not supported by ancestral sampling'
        ts = (t * (sde.N - 1) / sde.T).long()
        if ve:                                       # sampling.py:232-241
            sg = sde.discrete_sigmas[ts]
            adj = torch.where(ts == 0, torch.zeros_like(sg), sde.discrete_sigmas[ts - 1])
            d2 = sg ** 2 - adj ** 2
            a, b, c = torch.ones_like(sg), d2 * m, torch.sqrt(adj ** 2 * d2 / sg ** 2)
        else:                                        # sampling.py:243-251
            beta = sde.discrete_betas[ts]
            r = 1.0 / torch.sqrt(1. - beta)
            a, b, c = r, beta * r * m, torch.sqrt(beta)
    mean1, std_m = sde.marginal_prob(one, t)     # imputation: alpha*obs + std*z (sampling.py:415-416)
    coef = torch.zeros(t.numel(), L.COEF_STRIDE)
    coef[:, 0], coef[:, 1], coef[:, 2], coef[:, 3], coef[:, 4] = a, b, c, mean1[:, 0], std_m
    coef[:, 5] = m                               # score = raw * coef[5]  (the Langevin corrector's gradient)
    return coef, labels


def prior_scalars(sde, model, t, continuous=True):
    """Host scalars of the DPoser prior loss at one time t (python floats, fp32-evaluated)."""
    tt = torch.tensor([float(t)], dtype=torch.float32)
    alpha, sigma = sde.return_alpha_sigma(tt)
    if continuous or isinstance(sde, sde_lib.subVPSDE):
        labels = tt * 999
        std_score = sde.marginal_prob(torch.zeros(1, 1), tt)[1]
    else:
        labels = tt * (sde.N - 1)
        std_score = sde.sqrt_1m_alphas_cumprod[labels.long()]
    sig = sigma_at(model, labels)
    return dict(alpha=float(alpha.reshape(-1)[0]), std=float(sigma.reshape(-1)[0]), label=labels,
                inv_sigma_std=float(1.0 / (sig * std_score)))


def host_seed():
    """A 63-bit seed drawn from torch's global CPU generator (so torch.manual_seed controls the kernels' Philox)."""
    return int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())


def rot6d_needs_cuda(model, on_cuda, what):
    """A 126-D (rot6d) network runs ``what`` on the GPU only: refuse it, naming rot6d, before any library call."""
    if getattr(model, 'is_rot6d', False) and not on_cuda:
        raise NotImplementedError(f'{what} of rot6d (126-D) score networks runs on CUDA only: there is no CPU '
                                  'implementation (move the network to a CUDA device)')
