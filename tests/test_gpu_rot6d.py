"""GPU parity of the 126-D (rot6d) score network on both engines: forward, fused sampler (every predictor, imputation,
Langevin corrector fused and per-step), the balanced-schedule cut, the 126-column Philox layout, prior loss (+ DDIM),
completion and the SMPLify prior with a rot6d normaliser.  References: the float32 CPU oracle (oracle/score_ref.py),
whose forward is width-generic, with the synthetic weights built by its recipe at pose width 126."""
import ctypes as C
import types

import pytest
import torch

from conftest import max_rel, rel_err
from dposer_b200 import _lib as L
from dposer_b200 import misc, prior, sampling, sde_lib, synthetic, utils as mutils

pytestmark = pytest.mark.gpu
D = 126
ENGINES = [(L.ENGINE_FP32, 2e-5), (L.ENGINE_TC, 1e-3)]
SAMPLER_ENGINES = [(L.ENGINE_FP32, 5e-5), (L.ENGINE_TC, 1e-3)]


@pytest.fixture(scope='module')
def sd126():
    from oracle import score_ref
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(score_ref, 'POSE_D', D)
        return score_ref.make_state_dict(42)


@pytest.fixture(scope='module')
def m126():
    m = synthetic.make_score_model(42, pose_dim=6).cuda()
    yield m
    m.engine = L.ENGINE_AUTO


def _oracle_forward(sd, x, labels, chunk=8192):
    from oracle import score_ref as S
    return torch.cat([S.score_model_forward(sd, x[i:i + chunk], labels[i:i + chunk]) for i in range(0, len(x), chunk)])


def _rows_ok(out, ref, tol):
    """Whole-batch relative error <= tol and every row within 3 tol of its own largest value."""
    out, ref = out.double().cpu(), ref.double()
    row = (out - ref).abs().amax(1) / ref.abs().amax(1).clamp_min(1e-30)
    return rel_err(out, ref) <= tol and float(row.max()) <= 3 * tol, (rel_err(out, ref), float(row.max()))


@pytest.mark.parametrize('B', [1, 7, 127, 129, 500, 4096, 18944, 18945])
def test_forward_vs_oracle(m126, sd126, B):
    gen = torch.Generator().manual_seed(B)
    x = torch.randn(B, D, generator=gen)
    x[::11] *= 1e4                                       # rows at |x| ~ 1e4 exercise the bf16 hi / lo split
    out = torch.empty(B, D)
    for t in [1.0, 0.5, 0.1, 0.01, 1e-3]:
        lab = torch.full((B,), t * 999)
        ref = _oracle_forward(sd126, x, lab)
        for engine, tol in ENGINES:
            m126.engine = engine
            out = m126(x.cuda(), lab)
            ok, err = _rows_ok(out, ref, tol)
            assert ok, (B, t, engine, err)
    m126.engine = L.ENGINE_AUTO
    assert out.shape == (B, D)


def test_forward_per_row_time_vs_oracle(m126, sd126):
    B = 777
    gen = torch.Generator().manual_seed(3)
    x = torch.randn(B, D, generator=gen)
    lab = (torch.rand(B, generator=gen) * 999).floor()
    ref = _oracle_forward(sd126, x, lab)
    out = m126(x.cuda(), lab)                            # per-row labels: the fp32 engine
    ok, err = _rows_ok(out, ref, 2e-5)
    assert ok, err


def _run(m, engine, fn, **kw):
    m.engine = engine
    try:
        return fn(m, **kw)
    finally:
        m.engine = L.ENGINE_AUTO


@pytest.mark.parametrize('N,B', [(8, 256), (1000, 16)])
def test_em_sampler_vs_oracle(m126, sd126, N, B):
    from oracle import score_ref as S
    gen = torch.Generator().manual_seed(N)
    z0 = torch.randn(B, D, generator=gen)
    noise = torch.randn(N, 1, B, D, generator=gen)
    _, ref = S.pc_sample(sd126, S.SubVP(0.1, 20., N), z0, 1e-3, noise={i: {'pred': noise[i, 0]} for i in range(N)})
    cfg = synthetic.default_config()
    fn = sampling.get_sampling_fn(cfg, sde_lib.subVPSDE(0.1, 20., N), (B, D), lambda x: x, 1e-3, device='cuda')
    for engine, tol in SAMPLER_ENGINES:
        traj, out = _run(m126, engine, fn, z=z0, noise=noise.cuda())
        assert rel_err(out, ref) < (2e-4 if N == 1000 and engine == L.ENGINE_FP32 else tol), engine
        assert traj.shape == (N, B, D)


def test_completion_sampler_vs_oracle(m126, sd126):
    from oracle import score_ref as S
    B, N = 200, 8
    gen = torch.Generator().manual_seed(5)
    torch.manual_seed(5)
    poses = torch.randn(B, D, generator=gen) * 0.5
    mask, obs = misc.create_mask(poses, part='legs')
    assert int((mask[0] == 0).sum()) == 6 * len(misc.BodyPartIndices.legs)
    z0 = torch.randn(B, D, generator=gen)
    noise = torch.randn(N, 3, B, D, generator=gen)
    nz = {i: {'imp_c': noise[i, 0], 'pred': noise[i, 1], 'imp_p': noise[i, 2]} for i in range(N)}
    _, ref = S.pc_sample(sd126, S.SubVP(0.1, 20., N), z0, 1e-3, noise=nz, observation=obs, mask=mask, task='completion')
    cfg = synthetic.default_config()
    fn = sampling.get_sampling_fn(cfg, sde_lib.subVPSDE(0.1, 20., N), (B, D), lambda x: x, 1e-3, device='cuda')
    for engine, tol in SAMPLER_ENGINES:
        _, out = _run(m126, engine, fn, z=z0, noise=noise.cuda(), observation=obs, mask=mask,
                      args=types.SimpleNamespace(task='completion'))
        assert rel_err(out, ref) < tol, engine


@pytest.mark.parametrize('B,start', [(256, 992), (20000, 998)])
def test_langevin_sampler_vs_oracle(m126, sd126, B, start):
    """B = 256: the fused persistent kernel; B = 20000 (> 18 944 rows, more tiles than SMs): the per-step chain."""
    from oracle import score_ref as S
    N = 1000
    n = N - start
    gen = torch.Generator().manual_seed(B)
    z0 = torch.randn(B, D, generator=gen)
    noise = torch.randn(n, 2, B, D, generator=gen)
    nz = {start + i: {'corr': noise[i, 0], 'pred': noise[i, 1]} for i in range(n)}
    _, ref = S.pc_sample(sd126, S.SubVP(0.1, 20., N), z0, 1e-3, noise=nz, corrector='langevin', task='denoise',
                         start_step=start)
    cfg = synthetic.default_config()
    cfg.sampling.corrector = 'langevin'
    fn = sampling.get_sampling_fn(cfg, sde_lib.subVPSDE(0.1, 20., N), (B, D), lambda x: x, 1e-3, device='cuda')
    for engine, tol in SAMPLER_ENGINES:
        _, out = _run(m126, engine, fn, z=z0, noise=noise.cuda(), start_step=start,
                      args=types.SimpleNamespace(task='denoise'))
        assert rel_err(out, ref) < tol, (engine, rel_err(out, ref))


@pytest.mark.parametrize('pred', ['reverse_diffusion', 'ancestral_sampling'])
def test_vpsde_predictors_vs_table_chain(m126, sd126, pred):
    """The oracle has subVP only: the reference is the product's coefficient tables iterated on the CPU over the
    oracle's network output (as test_host_logic's chain test does against the real reference)."""
    from oracle import score_ref as S
    B, start, N = 96, 992, 1000
    sde = sde_lib.VPSDE(0.1, 20., N)
    ts = mutils.timestep_grid(sde, 1e-3)[start:]
    coef, labels = mutils.em_coefficients(sde, m126, ts, False, True, predictor=pred)
    gen = torch.Generator().manual_seed(11)
    z0 = torch.randn(B, D, generator=gen)
    noise = torch.randn(N - start, 1, B, D, generator=gen)
    x = z0.clone()
    for i in range(N - start):
        raw = S.score_model_forward(sd126, x, torch.ones(B) * labels[i], scale_by_sigma=False)
        xm = coef[i, 0] * x + coef[i, 1] * raw
        x = xm + coef[i, 2] * noise[i, 0]
    cfg = synthetic.default_config()
    cfg.sampling.predictor = pred
    fn = sampling.get_sampling_fn(cfg, sde, (B, D), lambda x: x, 1e-3, device='cuda')
    for engine, tol in SAMPLER_ENGINES:
        _, out = _run(m126, engine, fn, z=z0, noise=noise.cuda(), start_step=start,
                      args=types.SimpleNamespace(task='denoise'))
        assert rel_err(out, xm) < tol, engine


@pytest.mark.parametrize('task', ['none', 'completion'])
def test_balanced_schedule_matches_unsplit_run(m126, task):
    B, N, k = 40000, 6, (3 if task == 'completion' else 1)
    gen = torch.Generator().manual_seed(77)
    z0 = torch.randn(B, D, generator=gen)
    noise = torch.randn(N, k, B, D, generator=gen).cuda()
    kw = {}
    if task == 'completion':
        obs = torch.randn(B, D, generator=gen) * 0.3
        mask = (torch.rand(B, D, generator=gen) < 0.5).float()
        kw = dict(args=types.SimpleNamespace(task='completion'))
    cfg = synthetic.default_config()
    sde = sde_lib.subVPSDE(0.1, 20., N)
    m126.engine = L.ENGINE_TC
    try:
        def run(lo, hi):
            fn = sampling.get_sampling_fn(cfg, sde, (hi - lo, D), lambda x: x, 1e-3, device='cuda')
            extra = dict(kw)
            if task == 'completion':
                extra.update(observation=obs[lo:hi], mask=mask[lo:hi])
            traj, out = fn(m126, z=z0[lo:hi], noise=noise[:, :, lo:hi].contiguous(), **extra)
            return traj[-1], out
        full_last, full_out = run(0, B)
        for lo in range(0, B, 16384):
            hi = min(B, lo + 16384)
            last, out = run(lo, hi)
            assert torch.equal(out, full_out[lo:hi]), (task, lo)
            assert torch.equal(last, full_last[lo:hi]), (task, lo)
    finally:
        m126.engine = L.ENGINE_AUTO
    assert torch.isfinite(full_out).all()


def _fill(B, seed, step, slot):
    z = torch.empty(B, D, device='cuda')
    L.check(L.load().dpb_normal_fill_dim(L.ptr(z), B, C.c_uint64(seed), C.c_uint64(step), slot, D,
                                         L.current_stream(z.device)))
    return z


def test_philox_126_columns_are_independent_normals():
    B = 4096
    zs = torch.stack([_fill(B, 123, 7, s) for s in range(5)])          # [slot, B, 126]
    assert abs(float(zs.mean())) < 0.01 and abs(float(zs.std()) - 1) < 0.01
    assert abs(float((zs ** 4).mean()) - 3.0) < 0.1
    # every (slot, column) pair is its own stream: no two of the 630 columns are correlated (a shared counter gives 1)
    cols = zs.permute(1, 0, 2).reshape(B, -1).double()
    corr = torch.corrcoef(cols.T)
    off = corr - torch.eye(corr.shape[0], device=corr.device, dtype=corr.dtype)
    assert float(off.abs().max()) < 0.1
    for s in range(4):                                                 # the aliasing a 16-quad stride would give
        assert not torch.equal(zs[s, :, 64:124], zs[s + 1, :, :60])
    # the documented counter word slot * DP/4 + column/4: slot 1 of the 63-D layout (words 16..31) is slot 0, columns
    # 64.., of the 126-D layout -- the 63-D stream keeps its addressing (columns 0..61 of it; the 126-D row ends at 125)
    z63 = torch.empty(B, 63, device='cuda')
    L.check(L.load().dpb_normal_fill_dim(L.ptr(z63), B, C.c_uint64(123), C.c_uint64(7), 1, 63,
                                         L.current_stream(z63.device)))
    assert torch.equal(z63[:, :62], zs[0, :, 64:126])


def test_philox_one_step_table_returns_the_fill(m126):
    """a = 1, b = 0, c = 1 and x = 0: the sampler returns exactly its predictor draw (Philox slot 1, step offset)."""
    B = 300
    coef = torch.zeros(1, L.COEF_STRIDE)
    coef[0, 0], coef[0, 2], coef[0, 3] = 1.0, 1.0, 1.0
    table = m126.time_table(torch.tensor([500.0]))
    want = _fill(B, 99, 5, 1)
    for engine in (L.ENGINE_FP32, L.ENGINE_TC):
        x = torch.zeros(B, D, device='cuda')
        xm = torch.empty_like(x)
        sampling._run_steps(m126, x, coef.cuda(), table, None, None, None, 99, 5, None, xm, False, engine=engine)
        assert torch.equal(x, want), engine


def _prior_ref(sd, x0, t, z, weighted, reduce, divisor=None, multi=False):
    from oracle import score_ref as S
    return S.prior_loss(sd, S.SubVP(0.1, 20., 1000), x0, torch.tensor([t]).expand(x0.shape[0]), z, weighted, reduce,
                        divisor, multi_denoise=multi)


def _grad_close(g, ref, x0, tol, div):
    g, ref = g.double().cpu(), ref.double()
    floor = tol * 2.0 * float(x0.abs().max()) / div           # x0 - x0_hat cancels as t -> 0 (see test_gpu_prior)
    return float((g - ref).abs().max()) <= tol * float(ref.abs().max()) + floor


@pytest.mark.parametrize('engine,tol', [(L.ENGINE_FP32, 5e-5), (L.ENGINE_TC, 1e-3)])
def test_prior_loss_vs_oracle(m126, sd126, engine, tol):
    sde = sde_lib.subVPSDE(0.1, 20., 1000)
    ts = mutils.timestep_grid(sde, 1e-3)
    B = 300
    gen = torch.Generator().manual_seed(8)
    x0 = torch.randn(B, D, generator=gen) * 0.8
    m126.engine = engine
    try:
        comp = prior.DPoserComp(m126, sde, True, batch_size=B)
        mp = prior.MotionPrior(m126, sde, True, batch_size=7)
        for q in [400, 799, 998]:
            t = float(ts[q])
            z = torch.randn(B, D, generator=gen)
            for weighted in (False, True):
                x = x0.cuda().requires_grad_(True)                # divisor B*D (mean), DPoserComp
                loss = comp.loss(x, torch.ones(B, device='cuda') * t, weighted=weighted, z=z.cuda())
                loss.backward()
                ref, gref = _prior_ref(sd126, x0, t, z, weighted, 'mean')
                assert abs(float(loss) - float(ref)) <= 4 * tol * abs(float(ref)) + 1e-9, (q, weighted)
                assert _grad_close(x.grad, gref, x0, tol, B * D), (q, weighted)
                x = x0.cuda().requires_grad_(True)                # divisor batch_size, MotionPrior
                loss = mp.DPoser_loss(x, torch.ones(B, device='cuda') * t, weighted=weighted, z=z.cuda())
                loss.backward()
                ref, gref = _prior_ref(sd126, x0, t, z, weighted, 'sum', 7.0)
                assert abs(float(loss) - float(ref)) <= 4 * tol * abs(float(ref)) + 1e-9, (q, weighted)
                assert _grad_close(x.grad, gref, x0, tol, 7.0), (q, weighted)
        # DDIM multi_denoise (10 affine steps in one sampler run)
        z = torch.randn(B, D, generator=gen)
        x = x0.cuda().requires_grad_(True)
        loss = mp.DPoser_loss(x, torch.ones(B, device='cuda') * float(ts[450]), weighted=False, multi_denoise=True,
                              z=z.cuda())
        loss.backward()
        ref, gref = _prior_ref(sd126, x0, float(ts[450]), z, False, 'sum', 7.0, multi=True)
        assert max_rel(loss.detach(), ref) < 4 * tol
        assert _grad_close(x.grad, gref, x0, 2 * tol, 7.0)
    finally:
        m126.engine = L.ENGINE_AUTO


@pytest.mark.parametrize('engine,tol', [(L.ENGINE_FP32, 2e-3), (L.ENGINE_TC, 5e-3)])
def test_completion_optimize_vs_oracle(m126, sd126, engine, tol):
    from oracle import fitting_loops
    B, iters, spi = 12, 2, 4
    gen = torch.Generator().manual_seed(21)
    torch.manual_seed(21)
    poses = torch.randn(B, D, generator=gen) * 0.5
    mask, obs = misc.create_mask(poses, part='left_arm')
    zs = [torch.randn(B, D, generator=gen) for _ in range(iters * spi)]
    ref = fitting_loops.completion_optimize(sd126, obs, mask, zs, lr=0.1, sample_trun=5.0, iterations=iters,
                                            steps_per_iter=spi)
    m126.engine = engine
    try:
        comp = prior.DPoserComp(m126, sde_lib.subVPSDE(0.1, 20., 1000), True, batch_size=B)
        out = comp.optimize(obs.cuda(), mask.cuda(), time_strategy='3', lr=0.1, sample_trun=5.0, iterations=iters,
                            steps_per_iter=spi, z_list=zs)
    finally:
        m126.engine = L.ENGINE_AUTO
    assert out.shape == (B, D)
    err = float((out.cpu() - ref).norm() / (ref - obs).norm())
    assert err < tol, err


def test_dposer_forward_with_rot6d_normalizer(m126, sd126):
    """DPoser.forward converts axis-angle -> rot6d -> normalised in torch; the prior's gradient reaches the axis-angle
    pose through autograd.  The draw z is the library's Philox (slot 3, step 0) under the seed torch's generator gives."""
    B = 64
    sde = sde_lib.subVPSDE(0.1, 20., 1000)
    norm = misc.Posenormalizer(None, device='cuda', normalize=True, min_max=False, rot_rep='rot6d')
    args = types.SimpleNamespace(device=torch.device('cuda'), sde_N=1000)
    pri = prior.DPoser(batch_size=B, args=args, model=m126, sde=sde, normalizer=norm)
    gen = torch.Generator().manual_seed(4)
    pose = (torch.randn(B, 69, generator=gen) * 0.4).cuda().requires_grad_(True)
    quan_t = 700
    m126.engine = L.ENGINE_FP32
    try:
        torch.manual_seed(1234)
        loss = pri(pose, None, quan_t)
        loss.backward()
    finally:
        m126.engine = L.ENGINE_AUTO
    torch.manual_seed(1234)
    z = _fill(B, mutils.host_seed(), 0, 3).cpu()
    # reference: the oracle's loss and gradient w.r.t. the normalised rot6d pose, chained to the axis-angle pose by
    # autograd through the same torch conversion
    p = pose.detach().clone().requires_grad_(True)
    x0 = norm.offline_normalize(p[:, :63], from_axis=True)
    t = float(mutils.timestep_grid(sde, 1e-3)[quan_t])
    ref, g_x0 = _prior_ref(sd126, x0.detach().cpu(), t, z, True, 'sum', float(B))
    (g_pose,) = torch.autograd.grad(x0, p, g_x0.cuda())
    assert abs(float(loss) - float(ref)) <= 2e-4 * abs(float(ref))
    assert max_rel(pose.grad, g_pose) < 1e-3
    assert float(pose.grad[:, 63:].abs().max()) == 0.0
