"""GPU parity: fused PC sampler (EM predictor, imputation, PF-ODE, start_step, Langevin) with the
reference's Gaussian draws injected, against golden vectors produced by the real reference."""
import types

import numpy as np
import pytest
import torch

from conftest import golden, rel_err, max_rel
from dposer_b200 import _lib as L
from dposer_b200 import sampling, sde_lib, synthetic

pytestmark = pytest.mark.gpu
CASES = [('em8', 8, 'none', None, False, 0), ('em32', 32, 'none', None, False, 0),
         ('comp8', 8, 'none', 'completion', False, 0), ('ode8', 8, 'none', None, True, 0),
         ('den16', 16, 'none', 'denoise', False, 10), ('lang8', 1000, 'langevin', 'denoise', False, 992)]


def _noise(g, name, task, corr):
    planes = []
    if corr == 'langevin':
        planes.append(g[f'{name}_noise_corr'])
    if task == 'completion':
        planes += [g[f'{name}_noise_imp_c'], g[f'{name}_noise_pred'], g[f'{name}_noise_imp_p']]
    else:
        planes.append(g[f'{name}_noise_pred'])
    return torch.tensor(np.stack(planes, axis=1)).cuda().contiguous()          # [n, K, B, 63]


@pytest.mark.parametrize('engine,tol', [(L.ENGINE_FP32, 5e-5), (L.ENGINE_TC, 1e-3)])
@pytest.mark.parametrize('case', CASES, ids=[c[0] for c in CASES])
def test_pc_sampler_vs_reference_golden(gpu_model, case, engine, tol):
    name, N, corr, task, pf, start = case
    g = golden('sampler_golden.npz')
    cfg = synthetic.default_config()
    cfg.sampling.corrector = corr
    cfg.sampling.probability_flow = pf
    sde = sde_lib.subVPSDE(0.1, 20., N)
    B = g[f'{name}_z0'].shape[0]
    fn = sampling.get_sampling_fn(cfg, sde, (B, 63), lambda x: x, 1e-3, device='cuda')
    obs = torch.tensor(g[f'{name}_obs']) if f'{name}_obs' in g.files else None
    mask = torch.tensor(g[f'{name}_mask']) if f'{name}_mask' in g.files else None
    args = types.SimpleNamespace(task=task) if task else None
    gpu_model.engine = engine
    try:
        traj, out = fn(gpu_model, observation=obs, mask=mask, z=torch.tensor(g[f'{name}_z0']), start_step=start,
                       args=args, noise=_noise(g, name, task, corr))
    finally:
        gpu_model.engine = L.ENGINE_AUTO
    assert traj.shape == (N - start, B, 63)
    assert max_rel(out, g[f'{name}_out']) < tol, name
    assert max_rel(traj[-1], g[f'{name}_traj_last']) < tol, name


def test_sampler_1000_steps_vs_oracle(gpu_model, oracle_sd):
    """Full-length run (N=1000, EM, injected noise) on both engines: relative error of x_mean <= 1e-3."""
    from oracle import score_ref as S
    B, N = 16, 1000
    gen = torch.Generator().manual_seed(1234)
    z0 = torch.randn(B, 63, generator=gen)
    noise = torch.randn(N, 1, B, 63, generator=gen)
    _, ref = S.pc_sample(oracle_sd, S.SubVP(0.1, 20., N), z0, 1e-3, noise={i: {'pred': noise[i, 0]} for i in range(N)})
    cfg = synthetic.default_config()
    fn = sampling.get_sampling_fn(cfg, sde_lib.subVPSDE(0.1, 20., N), (B, 63), lambda x: x, 1e-3, device='cuda',
                                  return_trajs=False)
    for engine, tol in [(L.ENGINE_FP32, 2e-4), (L.ENGINE_TC, 1e-3)]:
        gpu_model.engine = engine
        try:
            traj, out = fn(gpu_model, z=z0, noise=noise.cuda())
        finally:
            gpu_model.engine = L.ENGINE_AUTO
        assert traj is None
        assert rel_err(out, ref) < tol, engine


def test_inkernel_philox_noise_is_standard_normal_and_engine_independent(gpu_model):
    import ctypes as C
    B = 4096
    z = torch.empty(B, 63, device='cuda')
    L.check(L.load().dpb_normal_fill_dim(L.ptr(z), B, C.c_uint64(123), C.c_uint64(7), 1, 63,
                                         L.current_stream(z.device)))
    assert abs(float(z.mean())) < 0.01 and abs(float(z.std()) - 1) < 0.01
    assert abs(float((z ** 4).mean()) - 3.0) < 0.1                      # kurtosis of N(0,1)
    z2 = torch.empty_like(z)
    L.check(L.load().dpb_normal_fill_dim(L.ptr(z2), B, C.c_uint64(123), C.c_uint64(8), 1, 63,
                                         L.current_stream(z.device)))
    assert abs(float((z * z2).mean())) < 0.01                           # steps are independent
    # same seed -> same samples on both engines (they share the Philox addressing)
    cfg = synthetic.default_config()
    fn = sampling.get_sampling_fn(cfg, sde_lib.subVPSDE(0.1, 20., 8), (256, 63), lambda x: x, 1e-3, device='cuda')
    z0 = torch.randn(256, 63)
    outs = []
    for engine in (L.ENGINE_FP32, L.ENGINE_TC):
        gpu_model.engine = engine
        torch.manual_seed(5)
        outs.append(fn(gpu_model, z=z0)[1])
    gpu_model.engine = L.ENGINE_AUTO
    assert rel_err(outs[1], outs[0]) < 1e-3


def test_completion_keeps_observed_dims_statistics(gpu_model):
    """Size-independent property of imputation: after the last step the trajectory state equals
    alpha*obs + std*z on observed dims (mask==1), so with std(t_last)~1e-4 it is ~obs."""
    cfg = synthetic.default_config()
    poses, mask, obs = synthetic.completion_inputs(n_partial=300, hypotheses=2)
    N = 50
    fn = sampling.get_sampling_fn(cfg, sde_lib.subVPSDE(0.1, 20., N), (600, 63), lambda x: x, 1e-3, device='cuda')
    traj, x_mean = fn(gpu_model, observation=obs, mask=mask, args=types.SimpleNamespace(task='completion'))
    last = traj[-1].cpu()
    sel = mask.bool()
    assert (last[sel] - obs[sel]).abs().max() < 5e-3


@pytest.mark.parametrize('task', ['none', 'completion'])
def test_sampler_balanced_schedule_matches_unsplit_run(gpu_model, task):
    """More row tiles than SMs: the fused sampler cuts step chains between CTA pairs (score_tc.cu: SegIter) and
    hands x over through x_io.  Rows are independent, so with injected noise the big run must equal, bit for bit,
    the same rows sampled in slices small enough that no chain is cut."""
    B, N, k = 40000, 6, (3 if task == 'completion' else 1)
    gen = torch.Generator().manual_seed(77)
    z0 = torch.randn(B, 63, generator=gen)
    noise = torch.randn(N, k, B, 63, generator=gen).cuda()
    kw = {}
    if task == 'completion':
        obs = torch.randn(B, 63, generator=gen) * 0.3
        mask = (torch.rand(B, 63, generator=gen) < 0.5).float()
        kw = dict(args=types.SimpleNamespace(task='completion'))
    cfg = synthetic.default_config()
    sde = sde_lib.subVPSDE(0.1, 20., N)
    gpu_model.engine = L.ENGINE_TC
    try:
        def run(lo, hi):
            fn = sampling.get_sampling_fn(cfg, sde, (hi - lo, 63), lambda x: x, 1e-3, device='cuda')
            extra = dict(kw)
            if task == 'completion':
                extra.update(observation=obs[lo:hi], mask=mask[lo:hi])
            traj, out = fn(gpu_model, z=z0[lo:hi], noise=noise[:, :, lo:hi].contiguous(), **extra)
            return traj[-1], out
        full_last, full_out = run(0, B)
        step = 16384
        for lo in range(0, B, step):
            hi = min(B, lo + step)
            last, out = run(lo, hi)
            assert torch.equal(out, full_out[lo:hi]), (task, lo)
            assert torch.equal(last, full_last[lo:hi]), (task, lo)
    finally:
        gpu_model.engine = L.ENGINE_AUTO
    assert torch.isfinite(full_out).all()


def test_ode_sampler_vs_oracle_rk45(gpu_model, oracle_sd):
    """Probability-flow ODE sampler (sampling.py:471-542): scipy RK45 on the host drives the drift evaluated by the
    GPU kernels; the same integrator driven by the oracle's drift is the reference.  The adaptive step control sees
    slightly different drifts, so the end points agree to the integrator's own accuracy, not to rounding."""
    from scipy import integrate
    from oracle import score_ref as S
    B = 16
    gen = torch.Generator().manual_seed(21)
    z0 = torch.randn(B, 63, generator=gen)
    osde = S.SubVP(0.1, 20., 1000)

    def rhs(t, xf):
        x = torch.tensor(xf, dtype=torch.float32).reshape(B, 63)
        d = S.reverse_drift(oracle_sd, osde, x, torch.ones(B) * float(t), probability_flow=True)[0]
        return d.reshape(-1).numpy()

    sol = integrate.solve_ivp(rhs, (1.0, 1e-3), z0.reshape(-1).numpy(), rtol=1e-5, atol=1e-5, method='RK45')
    ref = torch.tensor(sol.y[:, -1], dtype=torch.float32).reshape(B, 63)
    fn = sampling.get_ode_sampler(sde_lib.subVPSDE(0.1, 20., 1000), (B, 63), lambda x: x, eps=1e-3, device='cuda')
    for engine, tol in [(L.ENGINE_FP32, 2e-3), (L.ENGINE_TC, 5e-3)]:
        gpu_model.engine = engine
        try:
            nfe, x = fn(gpu_model, z=z0)
        finally:
            gpu_model.engine = L.ENGINE_AUTO
        assert rel_err(x, ref) < tol, (engine, float(rel_err(x, ref)))
        assert abs(nfe - sol.nfev) <= 0.25 * sol.nfev, (nfe, sol.nfev)


@pytest.mark.parametrize('engine,tol', [(L.ENGINE_FP32, 5e-5), (L.ENGINE_TC, 1e-3)])
def test_vpsde_em_sampler_vs_reference_golden(gpu_model, engine, tol):
    """Euler-Maruyama sampling under VPSDE (the fused kernel's affine step with VPSDE coefficients) against the real
    reference with replayed draws."""
    g = golden('sde_variants_golden.npz')
    N, B = 8, 5
    cfg = synthetic.default_config()
    fn = sampling.get_sampling_fn(cfg, sde_lib.VPSDE(0.1, 20., N), (B, 63), lambda x: x, 1e-3, device='cuda')
    noise = torch.tensor(g['vp_em_noise'])[:, None].cuda()
    gpu_model.engine = engine
    try:
        traj, out = fn(gpu_model, z=torch.tensor(g['vp_em_z0']), noise=noise)
    finally:
        gpu_model.engine = L.ENGINE_AUTO
    assert max_rel(out, g['vp_em_out']) < tol
    assert max_rel(traj[-1], g['vp_em_last']) < tol


def test_sampler_full_size_run_is_reproducible(gpu_model):
    """BASELINE.json's full size (65 536 poses, N = 1000) through a size-independent property: the same seed gives
    the same samples bit for bit (Philox is keyed by (row, step); the CTA pairs hand step chains over through global
    memory, so a missed hand-off or a race would show up here), and the samples are finite."""
    B, N = 65536, 1000
    cfg = synthetic.default_config()
    fn = sampling.get_sampling_fn(cfg, sde_lib.subVPSDE(0.1, 20., N), (B, 63), lambda x: x, 1e-3, device='cuda',
                                  return_trajs=False)
    z0 = torch.randn(B, 63, generator=torch.Generator().manual_seed(5))
    gpu_model.engine = L.ENGINE_TC
    try:
        outs = []
        for _ in range(2):
            torch.manual_seed(99)
            outs.append(fn(gpu_model, z=z0)[1])
    finally:
        gpu_model.engine = L.ENGINE_AUTO
    assert torch.isfinite(outs[0]).all()
    assert torch.equal(outs[0], outs[1])


@pytest.mark.parametrize('tag,sde_name,pred', [('vp_rd', 'vp', 'reverse_diffusion'), ('vp_anc', 'vp', 'ancestral_sampling'),
                                              ('sub_rd', 'subvp', 'reverse_diffusion')])
@pytest.mark.parametrize('engine,tol', [(L.ENGINE_FP32, 5e-5), (L.ENGINE_TC, 1e-3)])
def test_other_predictors_vs_reference_golden(gpu_model, tag, sde_name, pred, engine, tol):
    """ReverseDiffusion / AncestralSampling predictors (sampling.py:210-259) as coefficient tables of the fused sampler,
    against the REAL reference classes called step by step over the last 8 steps of the N = 1000 grid with replayed draws
    (sde_variants_golden.npz)."""
    import types
    g = golden('sde_variants_golden.npz')
    N, B = 1000, 5
    assert np.isfinite(g[f'{tag}_out']).all()
    cfg = synthetic.default_config()
    cfg.sampling.predictor = pred
    sde = sde_lib.VPSDE(0.1, 20., N) if sde_name == 'vp' else sde_lib.subVPSDE(0.1, 20., N)
    fn = sampling.get_sampling_fn(cfg, sde, (B, 63), lambda x: x, 1e-3, device='cuda')
    noise = torch.tensor(g[f'{tag}_noise'])[:, None].cuda()
    gpu_model.engine = engine
    try:
        traj, out = fn(gpu_model, z=torch.tensor(g['vp_em_z0']), noise=noise, start_step=N - 8,
                       args=types.SimpleNamespace(task='denoise'))
    finally:
        gpu_model.engine = L.ENGINE_AUTO
    assert max_rel(out, g[f'{tag}_out']) < tol
    assert max_rel(traj[-1], g[f'{tag}_last']) < tol


@pytest.mark.parametrize('tag,pred', [('ve_em', 'euler_maruyama'), ('ve_rd', 'reverse_diffusion'),
                                      ('ve_anc', 'ancestral_sampling')])
@pytest.mark.parametrize('engine,tol', [(L.ENGINE_FP32, 5e-5), (L.ENGINE_TC, 1e-3)])
def test_vesde_predictors_vs_reference_golden(gpu_model, tag, pred, engine, tol):
    """VESDE (sde_lib.py:234-295; score = +raw / sigma with labels = sigma(t), utils.py:164-180) through the three
    predictors as coefficient tables of the fused sampler: 8 steps from 50 z, draws replayed, against the REAL
    reference (its own pc_sampler for Euler-Maruyama, the predictor classes called directly for the other two)."""
    g = golden('sde_variants_golden.npz')
    N, B = 8, 5
    cfg = synthetic.default_config()
    cfg.sampling.predictor = pred
    sde = sde_lib.VESDE(0.01, 50., N)
    fn = sampling.get_sampling_fn(cfg, sde, (B, 63), lambda x: x, 1e-5, device='cuda')
    noise = torch.tensor(g[f'{tag}_noise'])[:, None].cuda()
    gpu_model.engine = engine
    try:
        traj, out = fn(gpu_model, z=torch.tensor(g['ve_em_z0']), noise=noise)
    finally:
        gpu_model.engine = L.ENGINE_AUTO
    assert max_rel(out, g[f'{tag}_out']) < tol
    assert max_rel(traj[-1], g[f'{tag}_last']) < tol


def test_likelihood_function_evaluation_vs_reference_golden(gpu_model):
    """One ODE function evaluation of the likelihood (drift + Hutchinson divergence, likelihood.py:26-37,58-66) against
    the REAL reference's autograd: dpb_score_jvp's eps . (J eps) is the reference's eps . (J^T eps)."""
    from dposer_b200 import likelihood
    g = golden('sde_variants_golden.npz')
    sde = sde_lib.subVPSDE(0.1, 20., 1000)
    drift, div = likelihood.drift_and_div(gpu_model, sde, torch.tensor(g['lik_xt']).cuda(), 0.3,
                                          torch.tensor(g['lik_eps']).cuda())
    assert max_rel(drift, g['lik_drift']) < 2e-5
    assert max_rel(div, g['lik_div']) < 2e-4


def test_likelihood_vs_reference_golden(gpu_model):
    """get_likelihood_fn (likelihood.py:40-113): bits/dim, latent code and function-evaluation count against the REAL
    reference on four AMASS poses with the same Rademacher probe (RK45 on the host on both sides)."""
    from dposer_b200 import likelihood
    g = golden('sde_variants_golden.npz')
    sde = sde_lib.subVPSDE(0.1, 20., 1000)
    fn = likelihood.get_likelihood_fn(sde, lambda v: v, rtol=1e-5, atol=1e-5, eps=1e-5)
    bpd, z, nfe = fn(gpu_model, torch.tensor(g['lik_data']).cuda(), epsilon=torch.tensor(g['lik_eps']).cuda())
    assert max_rel(bpd, g['lik_bpd']) < 2e-3
    assert max_rel(z, g['lik_z']) < 5e-3
    # device-side RK45 with scipy's controller: the step sequence follows the reference's to within a few evaluations
    assert abs(nfe - int(g['lik_nfe'])) <= 0.02 * int(g['lik_nfe']), (nfe, int(g['lik_nfe']))
