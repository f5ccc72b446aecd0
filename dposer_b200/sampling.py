"""Samplers with the reference's call surface (lib/algorithms/advanced/sampling.py).

``get_sampling_fn(config, sde, shape, inverse_scaler, eps, device)`` returns
``pc_sampler(model, observation, mask, z, start_step, args) -> (trajs, x)`` or
``ode_sampler(model, z) -> (nfe, x)`` exactly like the reference, but the hot loop
(sampling.py:456-461) is ONE call into libdposer_b200: ``dpb_sampler_run`` evaluates all
steps (score net + Euler-Maruyama update + imputation + noise) on the device; with the
tcgen05 engine that is a single persistent kernel.  The Langevin corrector needs batch-global
norms every step (sampling.py:296-297), so that variant runs step by step
(corrector kernels + a one-step ``dpb_sampler_run``).
"""
import ctypes as C

import numpy as np
import torch
from scipy import integrate

from . import _lib as L
from . import sde_lib
from . import utils as mutils

_PREDICTORS = ('euler_maruyama', 'reverse_diffusion', 'ancestral_sampling', 'none')
_CORRECTORS = ('none', 'langevin')


def get_sampling_fn(config, sde, shape, inverse_scaler, eps, device=None, return_trajs=True):
    """sampling.py:80-124.  ``return_trajs=False`` skips materialising the [N,B,63] trajectory
    (252 KB per row at N=1000) and returns ``None`` in its place."""
    if device is None:
        device = config.device
    name = config.sampling.method.lower()
    if name == 'ode':
        return get_ode_sampler(sde, shape, inverse_scaler, denoise=config.sampling.noise_removal, eps=eps,
                               device=device)
    if name == 'pc':
        pred, corr = config.sampling.predictor.lower(), config.sampling.corrector.lower()
        if pred not in _PREDICTORS:
            raise NotImplementedError(f'predictor {pred!r} is not supported')
        # reverse_diffusion / ancestral_sampling (sampling.py:210-259): the reference's own pc_sampler cannot drive them
        # (update_fn arity, sampling.py:215 vs :361 -- SURVEY 2 row 4); here they are two more coefficient tables of the
        # same fused kernel, pinned against the reference classes called directly (sde_variants_golden.npz)
        if pred == 'ancestral_sampling' and not isinstance(sde, (sde_lib.VPSDE, sde_lib.VESDE)):
            raise NotImplementedError(f'SDE class {sde.__class__.__name__} not yet supported.')   # sampling.py:229
        if corr not in _CORRECTORS:
            raise NotImplementedError(f'corrector {corr!r} is not supported')
        return get_pc_sampler(sde, shape, pred, corr, inverse_scaler, config.sampling.snr,
                              n_steps=config.sampling.n_steps_each,
                              probability_flow=config.sampling.probability_flow,
                              continuous=config.training.continuous, denoise=config.sampling.noise_removal,
                              eps=eps, device=device, return_trajs=return_trajs)
    raise ValueError(f"Sampler name {name} unknown.")


def _run_steps(model, x, coef, table, obs, mask, noise, seed, step_offset, traj, x_mean, impute, engine=None):
    """One dpb_sampler_run over the rows of ``coef`` (device fp32 [n,8]) / ``table`` ([n,5,1024])."""
    model.check_width(x, 'x')
    h = model.handle()
    B = x.shape[0]
    tbl = L.StepTables(coef.shape[0], C.c_void_p(coef.data_ptr()), C.c_void_p(table.data_ptr()))
    flags = model.engine if engine is None else engine
    if impute:
        flags |= L.SAMPLER_IMPUTE
    if noise is not None:
        flags |= L.SAMPLER_NOISE_GIVEN
    ws = model.workspace(B, x.device)
    L.check(L.load().dpb_sampler_run(h.ptr, L.ptr(x), C.byref(tbl), L.ptr(obs), L.ptr(mask), L.ptr(noise),
                                     C.c_uint64(seed), C.c_uint64(step_offset), L.ptr(traj), L.ptr(x_mean), B, flags,
                                     L.ptr(ws), ws.numel(), L.current_stream(x.device)))


def get_pc_sampler(sde, shape, predictor, corrector, inverse_scaler, snr, n_steps=1, probability_flow=False,
                   continuous=False, denoise=True, eps=1e-3, device='cuda', return_trajs=True):
    """sampling.py:375-468."""
    if n_steps != 1 and corrector != 'none':
        raise NotImplementedError('n_steps_each != 1 is not supported (shipped config uses 1)')
    device = torch.device(device)

    def pc_sampler(model, observation=None, mask=None, z=None, start_step=0, args=None, noise=None):
        """``noise`` (optional, parity mode): device tensor [N-start, K, B, D] of the Gaussian draws in the
        reference's order -- K=1 (predictor) or K=3 with completion (after-corrector, predictor, after-predictor)."""
        with torch.no_grad():
            if len(shape) != 2 or shape[1] != model.pose_width:
                raise ValueError(f'sampler shape {tuple(shape)} does not match the {model.pose_width}-D score network')
            task = getattr(args, 'task', None) if args is not None else None
            impute = task == 'completion'
            start_t = start_step if task == 'denoise' else 0
            n_run = sde.N - start_t
            if z is not None:
                model.check_width(z, 'z')
            B = shape[0] if z is None else z.shape[0]
            if impute:
                model.check_width(observation, 'observation', B)
                model.check_width(mask, 'mask', B)
            if noise is not None:
                # [n, K, B, D]: K = 1 predictor draw (+2 imputation draws) (+1 Langevin draw first)
                k = (3 if impute else 1) + (0 if corrector == 'none' else 1)
                if noise.dim() != 4 or noise.shape[0] < n_run or tuple(noise.shape[1:]) != (k, B, model.pose_width):
                    raise ValueError(f'noise: expected [>= {n_run}, {k}, {B}, {model.pose_width}], got {list(noise.shape)}')
                noise = noise.contiguous()
            if device.type != 'cuda':
                raise RuntimeError('dposer_b200 samplers run on CUDA only (no CPU fallback)')
            x = (sde.prior_sampling(shape) if z is None else z).to(device=device, dtype=torch.float32).contiguous()
            if z is not None:
                x = x.clone()
            timesteps = mutils.timestep_grid(sde, eps)
            if predictor == 'none':
                raise NotImplementedError("predictor 'none' (corrector-only sampling) is not supported")
            coef, labels = mutils.em_coefficients(sde, model, timesteps[start_t:], probability_flow, continuous,
                                                  predictor=predictor)
            coef = coef.to(device)
            table = model.time_table(labels)
            if impute:
                observation = observation.to(device=device, dtype=torch.float32).contiguous()
                mask = mask.to(device=device, dtype=torch.float32).contiguous()
            trajs = torch.empty(n_run, B, shape[1], device=device) if return_trajs else None
            x_mean = torch.empty_like(x)
            seed = mutils.host_seed() if noise is None else 0
            if n_run <= 0:
                return trajs, x
            if corrector == 'none':
                _run_steps(model, x, coef, table, observation, mask, noise, seed, start_t, trajs, x_mean, impute)
            else:
                _langevin_loop(model, sde, x, coef, table, timesteps[start_t:], observation, mask, noise, seed,
                               start_t, trajs, x_mean, impute, snr, continuous)
            return trajs, (x_mean if denoise else x)

    return pc_sampler


def _langevin_loop(model, sde, x, coef, table, t_run, obs, mask, noise, seed, start_t, trajs, x_mean, impute, snr,
                   continuous=True):
    """corrector -> (impute) -> predictor -> (impute) per step, sampling.py:459-460 with :282-302: ONE native call
    (``dpb_sampler_run_pc`` issues the five launches of every step itself).  Given-noise layout here is
    [n, K+1, B, 63] with the Langevin draw first."""
    lib = L.load()
    B = x.shape[0]
    dev = x.device
    if isinstance(sde, (sde_lib.VPSDE, sde_lib.subVPSDE)):
        lang_alpha = sde.alphas[(t_run * (sde.N - 1) / sde.T).long()]      # sampling.py:287-289
    else:
        lang_alpha = torch.ones_like(t_run)
    # same score scaling as the predictor (utils.get_score_fn: continuous marginal std, or the discrete VPSDE table),
    # evaluated for all steps at once by em_coefficients (column 5)
    scale = coef[:, 5].detach().to('cpu', torch.float32).contiguous()
    lang_alpha = lang_alpha.to(torch.float32).contiguous()
    h = model.handle()
    ws = torch.empty(int(lib.dpb_sampler_pc_workspace_bytes(h.ptr, B)), dtype=torch.uint8, device=dev)
    n = t_run.numel()
    tbl = L.StepTables(n, C.c_void_p(coef.data_ptr()), C.c_void_p(table.data_ptr()))
    flags = model.engine | (L.SAMPLER_IMPUTE if impute else 0) | (L.SAMPLER_NOISE_GIVEN if noise is not None else 0)
    nz = None if noise is None else noise.contiguous()
    L.check(lib.dpb_sampler_run_pc(h.ptr, L.ptr(x), C.byref(tbl), C.c_void_p(scale.data_ptr()),
                                   C.c_void_p(lang_alpha.data_ptr()), float(snr), L.ptr(obs), L.ptr(mask), L.ptr(nz),
                                   C.c_uint64(seed), C.c_uint64(start_t), L.ptr(trajs), L.ptr(x_mean), B, flags,
                                   L.ptr(ws), ws.numel(), L.current_stream(dev)))


def get_ode_sampler(sde, shape, inverse_scaler, denoise=False, rtol=1e-5, atol=1e-5, method='RK45', eps=1e-3,
                    device='cuda'):
    """sampling.py:471-542.  ``method='RK45'`` (the reference's default) integrates on the device (ode.py: scipy's step-size
    controller on the host, native stage / error kernels, fp64 state); other methods run scipy on the host over the GPU drift."""
    device = torch.device(device)

    def drift_fn(model, x, t):
        score_fn = mutils.get_score_fn(sde, model, train=False, continuous=True)
        return sde.reverse(score_fn, probability_flow=True).sde(x, t)[0]

    def ode_sampler(model, z=None):
        if method == 'RK45' and device.type == 'cuda' and getattr(model, 'is_rot6d', False):
            raise NotImplementedError('the device RK45 probability-flow ODE is built for the 63-D axis network, not for '
                                      'rot6d (126-D) score networks')
        with torch.no_grad():
            x = (sde.prior_sampling(shape) if z is None else z).to(device)
            if method == 'RK45' and device.type == 'cuda':
                # device-side Dormand-Prince (ode.py): fp64 state on the GPU, one scalar read back per attempted step
                from . import ode
                be = ode.PFOdeBackend(model, sde, x.to(torch.float32))
                nfev, _ = ode.solve_rk45(be, sde.T, eps, rtol=rtol, atol=atol)
                x = be.y.view(shape).to(torch.float32)
            else:
                def ode_func(t, xf):
                    xx = mutils.from_flattened_numpy(xf, shape).to(device).type(torch.float32)
                    vec_t = torch.ones(shape[0], device=device) * t
                    return mutils.to_flattened_numpy(drift_fn(model, xx, vec_t))

                sol = integrate.solve_ivp(ode_func, (sde.T, eps), mutils.to_flattened_numpy(x), rtol=rtol, atol=atol,
                                          method=method)
                nfev = sol.nfev
                x = torch.tensor(sol.y[:, -1]).reshape(shape).to(device).type(torch.float32)
            if denoise:
                # one reverse-diffusion predictor step without noise (sampling.py:492-499)
                vec_eps = torch.ones(x.shape[0], device=device) * eps
                score_fn = mutils.get_score_fn(sde, model, train=False, continuous=True)
                f, G = sde.reverse(score_fn, probability_flow=False).discretize(x, vec_eps)
                x = x - f
            return nfev, inverse_scaler(x)

    return ode_sampler
