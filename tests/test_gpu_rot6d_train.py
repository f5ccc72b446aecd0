"""GPU parity of the 126-D (rot6d) score network's training step, likelihood and device RK45 ODE sampler: three
get_step_fn steps against oracle/train_ref.py, the Philox z layout, the graphed and data-parallel steps, the forward /
backward halves, the score-network JVP on both paths and the probability-flow ODE against scipy over the oracle.
References: the CPU oracle with its weights recipe at pose width 126 (the 63-D tests' tolerances throughout)."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import max_rel, rel_err
from dposer_b200 import _lib as L
from dposer_b200 import likelihood, losses, misc, sampling, sde_lib, synthetic
from dposer_b200.ema import ExponentialMovingAverage

pytestmark = pytest.mark.gpu
D = 126


@pytest.fixture(scope='module')
def sd126():
    from oracle import score_ref
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(score_ref, 'POSE_D', D)
        return score_ref.make_state_dict(42)


def _state(cfg, model):
    opt = losses.get_optimizer(cfg, model.parameters())
    ema = ExponentialMovingAverage(model.parameters(), decay=cfg.model.ema_rate)
    return dict(optimizer=opt, model=model, ema=ema, step=0)


def _draws(B, seed):
    gen = torch.Generator().manual_seed(seed)
    t = torch.rand(B, generator=gen) * (1 - 1e-5) + 1e-5
    z = torch.randn(B, D, generator=gen)
    masks = (torch.rand(5, B, 1024, generator=gen) >= 0.1).to(torch.uint8)
    return t, z, masks


def _data(B, seed=0):
    return torch.randn(B, D, generator=torch.Generator().manual_seed(seed)) * 0.8


def test_train_steps_vs_oracle(sd126):
    """Three get_step_fn(train=True) steps (dropout 0.1, warm-up, clipping, Adam, EMA) with t, z and the dropout masks
    replayed, B = 200 (two 128-row tiles, not a multiple of 64): loss, gradients and their norm after every step;
    parameter / EMA / Adam-moment deltas at the end; then the evaluation step and two loss variants."""
    from oracle import score_ref as S
    from oracle import train_ref as T
    B, STEPS = 200, 3
    cfg = synthetic.default_config()
    model = synthetic.make_score_model(42, pose_dim=6).cuda()
    model.train()
    p0 = {n: p.detach().clone() for n, p in model.named_parameters()}
    state = _state(cfg, model)
    state['step'] = 2500                                   # half-way through the warm-up
    sde, osde = sde_lib.subVPSDE(0.1, 20., 1000), S.SubVP(0.1, 20., 1000)
    step_fn = losses.get_step_fn(sde, train=True, optimize_fn=losses.optimization_manager(cfg), reduce_mean=True)
    osd = {k: v.clone() for k, v in sd126.items()}
    names = T.param_names(osd)
    used = [k for k in names if not k.startswith('pre_dense_cond')]
    oopt = {k: (torch.zeros_like(osd[k]), torch.zeros_like(osd[k])) for k in used}
    oopt['step'] = 0
    oema = {k: osd[k].clone() for k in names}
    oema['num_updates'] = 0
    gmin = {}                     # per element: min over the steps of |g| / max |g| of its tensor (oracle gradients)
    for s in range(STEPS):
        batch = _data(B, s)
        t, z, masks = _draws(B, 100 + s)
        ld = step_fn(state, batch.cuda(), t=t, z=z, drop_mask=masks)
        oloss, og, onorm = T.train_step(osd, oopt, oema, osde, batch, t, z, masks, 2500 + s, p=0.1, lr=cfg.optim.lr,
                                        warmup=cfg.optim.warmup, grad_clip=cfg.optim.grad_clip,
                                        ema_rate=cfg.model.ema_rate)
        assert abs(float(ld['step_loss']) - float(oloss)) < 2e-4 * float(oloss), s
        assert abs(state['optimizer'].grad_norm() - float(onorm)) < 2e-4 * float(onorm), s
        for n, p in model.named_parameters():
            if n.startswith('pre_dense_cond'):
                assert float(p.grad.abs().max()) == 0.0
                continue
            assert p.grad.shape == og[n].shape
            assert max_rel(p.grad, og[n]) < 3e-4, (s, n)
            r = og[n].abs() / og[n].abs().max()
            gmin[n] = r if s == 0 else torch.minimum(gmin[n], r)
    assert state['step'] == 2500 + STEPS and state['ema'].num_updates == STEPS
    opt = state['optimizer']
    for i, (n, p) in enumerate(model.named_parameters()):
        if n.startswith('pre_dense_cond'):
            continue
        d, od = (p.detach() - p0[n]).cpu(), osd[n] - sd126[n]
        dmax = max(float(od.abs().max()), 1e-12)
        # Adam's step is +-lr for any gradient size, so an element whose gradient is at the level of the accepted gradient
        # error (3e-4 of the tensor's max) can take either sign: element by element, the deltas are compared where every
        # step's gradient is >= 1e-2 of its tensor's max (with gradients perturbed by the full accepted error, the
        # oracle's own deltas move by <= 1.7e-2 of the largest delta there); the norm over every element
        ok = gmin[n] >= 1e-2
        assert bool(ok.any()), n
        assert float((d - od)[ok].abs().max()) < 3e-2 * dmax + 1e-9, n
        assert abs(float(d.double().norm()) - float(od.double().norm())) < 1e-2 * float(od.double().norm()) + 1e-12, n
        e = (state['ema'].shadow_params[i] - p0[n]).cpu()
        assert float((e - (oema[n] - sd126[n]))[ok].abs().max()) < 3e-2 * dmax + 1e-9, n
        st = opt.state[p]
        m, v = oopt[n]
        assert float((st['exp_avg'].cpu() - m).abs().max()) < 3e-4 * float(m.abs().max()), n
        assert float((st['exp_avg_sq'].cpu() - v).abs().max()) < 6e-4 * float(v.abs().max()), n
    # ---- evaluation step: EMA weights, no dropout, parameters restored afterwards
    model.eval()
    before = [p.detach().clone() for p in model.parameters()]
    batch = _data(B, 9)
    t, z, _ = _draws(B, 9)
    eval_fn = losses.get_step_fn(sde, train=False, reduce_mean=True)
    ld = eval_fn(state, batch.cuda(), t=t, z=z)
    esd = dict(osd)
    esd.update({k: oema[k] for k in names})
    ref = T.sde_loss(esd, osde, batch, t, z, reduce_mean=True)
    assert abs(float(ld['step_loss']) - float(ref)) < 3e-4 * float(ref)
    assert all(torch.equal(a, p.detach()) for a, p in zip(before, model.parameters()))
    # ---- likelihood weighting and reduce_mean=False on the updated weights, with gradients
    model.config.model.dropout = 0.0
    try:
        for rm, lw in ((True, True), (False, False)):
            leaves = {k: osd[k].clone().requires_grad_(True) for k in used}
            full = dict(osd)
            full.update(leaves)
            ol = T.sde_loss(full, osde, batch, t, z, reduce_mean=rm, likelihood_weighting=lw)
            og = dict(zip(used, torch.autograd.grad(ol, [leaves[k] for k in used])))
            fn = losses.get_sde_loss_fn(sde, True, reduce_mean=rm, likelihood_weighting=lw)
            loss = fn(model, batch.cuda(), None, None, t=t, z=z)
            assert abs(float(loss) - float(ol)) < 3e-4 * abs(float(ol)), (rm, lw)
            for n, p in model.named_parameters():
                if n in og:
                    assert max_rel(p.grad, og[n]) < 5e-4, (rm, lw, n)
    finally:
        model.config.model.dropout = 0.1


def _fill(B, seed):
    z = torch.empty(B, D, device='cuda')
    L.check(L.load().dpb_normal_fill_dim(L.ptr(z), B, C.c_uint64(seed), C.c_uint64(0), 0, D, L.current_stream(z.device)))
    return z


def test_philox_z_is_the_126_column_layout():
    """A step without given draws: deterministic for a seed; its z is Philox keyed by (seed, row, counter = column quad),
    i.e. dpb_normal_fill_dim(seed, step 0, slot 0) (columns 64..127 from counters 16..31); those 126 columns are standard
    normal and columns 0..63 are uncorrelated with columns 64..127."""
    B = 4096
    model = synthetic.make_score_model(42, pose_dim=6).cuda()
    model.train()
    sde = sde_lib.subVPSDE(0.1, 20., 1000)
    fn = losses.get_sde_loss_fn(sde, True, reduce_mean=True)
    batch = _data(B).cuda()
    rows = fn.make_rows(model, B, torch.rand(B, generator=torch.Generator().manual_seed(3)) * 0.9 + 0.05)
    runs = []
    for z in (None, None, _fill(B, 77)):
        loss = losses.native_loss(model, batch, rows, z=z, drop_p=0.0, seed=77)
        g = torch.cat([p.grad.reshape(-1) for p in model.parameters()])
        runs.append((float(loss), g.clone()))
    assert np.isfinite(runs[0][0])
    for r in runs[1:]:
        assert r[0] == runs[0][0] and torch.equal(r[1], runs[0][1])
    assert float(losses.native_loss(model, batch, rows, drop_p=0.0, seed=78)) != runs[0][0]
    z = _fill(B, 77).double()
    assert float(z.mean(0).abs().max()) < 0.07 and float((z.var(0) - 1).abs().max()) < 0.1
    corr = torch.corrcoef(z.T)
    assert float(corr[:64, 64:].abs().max()) < 0.08
    assert not torch.equal(z[:, 64:124], z[:, :60])


def test_graphed_and_data_parallel_steps_match_eager():
    """get_step_fn(graph=True) replays the eager 126-D step bit for bit over several steps (two batch sizes, warm-up,
    EMA schedule); data_parallel=True in a single process (the all-reduce is the identity) does too."""
    cfg = synthetic.default_config()
    cfg.optim.warmup = 4
    sde = sde_lib.subVPSDE(0.1, 20., 1000)
    data = _data(320, 4).cuda()
    res = []
    for mode in ('eager', 'graph', 'dp'):
        model = synthetic.make_score_model(42, pose_dim=6).cuda()
        model.train()
        state = _state(cfg, model)
        step_fn = losses.get_step_fn(sde, train=True, optimize_fn=losses.optimization_manager(cfg), reduce_mean=True,
                                     graph=mode == 'graph', data_parallel=mode == 'dp')
        torch.manual_seed(5)
        ls = [float(step_fn(state, data[:160] if i % 2 else data)['step_loss']) for i in range(6)]
        res.append((ls, state['optimizer'].flat_p.clone(), state['ema']._flat.clone(), state['optimizer'].flat_m.clone(),
                    state['step'], state['ema'].num_updates, state['optimizer']._step))
    a = res[0]
    for b in res[1:]:
        assert a[0] == b[0], (a[0], b[0])
        assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])
        assert a[4:] == b[4:] == (6, 6, 6)


def test_sampler_network_after_a_step_is_the_oracle_on_the_new_weights():
    from oracle import score_ref as S
    cfg = synthetic.default_config()
    cfg.optim.warmup = 0
    model = synthetic.make_score_model(42, pose_dim=6).cuda()
    model.train()
    state = _state(cfg, model)
    sde = sde_lib.subVPSDE(0.1, 20., 1000)
    x, lab = torch.randn(5, D, generator=torch.Generator().manual_seed(1)).cuda(), torch.full((5,), 300.)
    model.eval()
    before = model(x, lab).clone()
    model.train()
    step_fn = losses.get_step_fn(sde, train=True, optimize_fn=losses.optimization_manager(cfg), reduce_mean=True)
    torch.manual_seed(2)
    step_fn(state, _data(200).cuda())
    model.eval()
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    for engine, tol in ((L.ENGINE_FP32, 2e-5), (L.ENGINE_TC, 1e-3)):
        model.engine = engine
        after = model(x, lab)
        assert float((after - before).abs().max()) > 0
        assert max_rel(after, S.score_model_forward(sd, x.cpu(), lab)) < tol, engine
    model.engine = L.ENGINE_AUTO


def test_forward_backward_halves_vs_autograd(sd126):
    """dpb_train_forward / dpb_train_backward (the halves the auxiliary loss chains) at 126: the output and the input
    cotangent g_in against autograd through oracle.train_ref.forward_train; the gradients too."""
    from oracle import train_ref as T
    B = 200
    model = synthetic.make_score_model(42, pose_dim=6).cuda()
    model.train()
    gen = torch.Generator().manual_seed(8)
    x = torch.randn(B, D, generator=gen)
    labels = torch.rand(B, generator=gen) * 999
    g_res = torch.randn(B, D, generator=gen)
    masks = (torch.rand(5, B, 1024, generator=gen) >= 0.1).to(torch.uint8)
    names = T.param_names(sd126)
    used = [k for k in names if not k.startswith('pre_dense_cond')]
    leaves = {k: sd126[k].clone().requires_grad_(True) for k in used}
    full = dict(sd126)
    full.update(leaves)
    xl = x.clone().requires_grad_(True)
    ref = T.forward_train(full, xl, labels, masks, 0.1, scale_by_sigma=False)
    grads = torch.autograd.grad((ref * g_res).sum(), [xl] + [leaves[k] for k in used])
    og_x, og = grads[0], dict(zip(used, grads[1:]))
    eng = losses._Engine(model, B, torch.device('cuda'))
    for p in model.parameters():
        p.grad = torch.zeros_like(p)
    P = losses._tensor_struct(model, lambda p: p.data)
    P.emb_freqs = losses._f32p(eng.freqs)
    G = losses._tensor_struct(model, lambda p: p.grad)
    lib, st = L.load(), L.current_stream(torch.device('cuda'))
    xd, ld, md, gd = x.cuda(), labels.cuda(), masks.cuda(), g_res.cuda()
    res = torch.empty(B, D, device='cuda')
    g_x = torch.empty(B, D, device='cuda')
    L.check(lib.dpb_train_forward(eng.ptr, C.byref(P), L.ptr(xd), L.ptr(ld), L.ptr(md), 0.1, C.c_uint64(0), L.ptr(res), st))
    L.check(lib.dpb_train_backward(eng.ptr, C.byref(P), C.byref(G), L.ptr(gd), L.ptr(md), 0.1, C.c_uint64(0), 0,
                                   L.ptr(g_x), st))
    torch.cuda.synchronize()
    assert max_rel(res, ref.detach()) < 2e-4
    assert max_rel(g_x, og_x) < 3e-4
    for n, p in model.named_parameters():
        if n in og:
            assert max_rel(p.grad, og[n]) < 5e-4, n


def _fwd64(sd, x, labels):
    """oracle.score_ref.score_model_forward in float64 (the time embedding's fp32 sin / cos widened)."""
    from oracle import score_ref as S
    import torch.nn.functional as F
    temb = F.silu(S._lin(sd, 'shared_time_embed.0', S.timestep_embedding(labels).double()))
    h = F.silu(S._gn(sd, 'pre_gnorm', S._lin(sd, 'pre_dense', x) + S._lin(sd, 'pre_dense_t', temb)))
    for b in (1, 2):
        h1 = F.silu(S._gn(sd, f'b{b}_gnorm1', S._lin(sd, f'b{b}_dense1', h) + S._lin(sd, f'b{b}_dense1_t', temb)))
        h2 = F.silu(S._gn(sd, f'b{b}_gnorm2', S._lin(sd, f'b{b}_dense2', h1) + S._lin(sd, f'b{b}_dense2_t', temb)))
        h = h + h2
    return S._lin(sd, 'post_dense', h) / sd['sigmas'][labels.long()].reshape(-1, 1)


def _schedule(t, n):
    """(f_x, g^2, std) of the sub-VP SDE at time t for n rows, as the reference evaluates them: fp32 torch scalars (the
    oracle's SubVP), widened to float64.  std = 1 - exp(2 lmc) cancels at small t, so its fp32 value is part of the
    reference's definition (at t = 1e-3 it differs from the float64 value by ~2.5e-4)."""
    from oracle import score_ref as S
    osde = S.SubVP(0.1, 20., 1000)
    tt = torch.full((n,), float(t))
    fx = osde.sde(torch.ones(n, 1), tt)[0][:, 0]
    g = osde.sde(torch.zeros(n, 1), tt)[1]
    std = osde.marginal(torch.zeros(n, 1), tt)[1]
    return fx.double(), (g ** 2).double(), std.double(), tt


def _score64(sd64, x, t):
    """score = -net(x, 999 t) / std(t): the network in float64, the schedule scalars as the reference computes them."""
    _, _, std, tt = _schedule(t, x.shape[0])
    return -_fwd64(sd64, x, tt * 999) / std[:, None]


def _drift_div64(sd64, x, eps, t):
    """Probability-flow drift and eps . (J_drift eps), float64 autograd through the oracle network (sub-VP, beta 0.1 .. 20)."""
    fx, g2, _, _ = _schedule(t, x.shape[0])
    xl = x.double().clone().requires_grad_(True)
    score = _score64(sd64, xl, t)
    drift = fx[:, None] * xl - 0.5 * g2[:, None] * score
    e = eps.double()
    div = (torch.autograd.grad((drift * e).sum(), xl)[0] * e).sum(1)
    return drift.detach(), div, score.detach()


@pytest.mark.parametrize('B', [1, 127, 129, 4097])
def test_score_jvp_vs_float64(sd126, B):
    """likelihood.drift_and_div (batch-uniform t: the tcgen05 JVP) and dpb_score_jvp with a per-row t_index (the fp32
    JVP) at 126 against float64 autograd through the oracle network: drift / score <= 2e-5, divergence <= 2e-4."""
    from dposer_b200 import utils as mutils
    model = synthetic.make_score_model(42, pose_dim=6).cuda()
    sd64 = {k: v.double() for k, v in sd126.items()}
    sde = sde_lib.subVPSDE(0.1, 20., 1000)
    gen = torch.Generator().manual_seed(B)
    x = torch.randn(B, D, generator=gen)
    eps = torch.randint(0, 2, (B, D), generator=gen).float() * 2 - 1
    ts = [1e-3, 0.3, 1.0]
    for t in ts:
        drift, div = likelihood.drift_and_div(model, sde, x.cuda(), t, eps.cuda())
        rd, rdiv, _ = _drift_div64(sd64, x, eps, t)
        assert max_rel(drift, rd) < 2e-5, t
        assert max_rel(div, rdiv) < 2e-4, t
    # per-row time: rows cycle through the three times; out = score, jv . eps = eps . (J_score eps)
    tt = torch.tensor(ts, dtype=torch.float32)
    coef, labels = mutils.em_coefficients(sde, model, tt, probability_flow=True, continuous=True)
    idx = torch.arange(B) % 3
    table = model.time_table(labels)
    h = model.handle()
    lib = L.load()
    ws = torch.empty(int(lib.dpb_score_jvp_workspace_bytes(h.ptr, B)), dtype=torch.uint8, device='cuda')
    xd, ed = x.cuda(), eps.cuda()
    ti = idx.to(torch.int32).cuda()
    rs = coef[idx, 5].float().contiguous().cuda()
    out, jv = torch.empty(B, D, device='cuda'), torch.empty(B, D, device='cuda')
    L.check(lib.dpb_score_jvp(h.ptr, L.ptr(xd), L.ptr(ed), L.ptr(table), L.ptr(ti), L.ptr(rs), 1.0, L.ptr(out), L.ptr(jv),
                              B, L.ptr(ws), ws.numel(), L.current_stream(xd.device)))
    ref_s, ref_q = torch.empty(B, D, dtype=torch.float64), torch.empty(B, dtype=torch.float64)
    for k, t in enumerate(ts):
        rows = idx == k
        if not rows.any():
            continue
        xl = x[rows].double().clone().requires_grad_(True)
        score = _score64(sd64, xl, t)
        e = eps[rows].double()
        ref_q[rows] = (torch.autograd.grad((score * e).sum(), xl)[0] * e).sum(1)
        ref_s[rows] = score.detach()
    assert max_rel(out, ref_s) < 2e-5
    assert max_rel((jv * ed).sum(1), ref_q) < 2e-4


def _rot6d_poses(n):
    from dposer_b200.transforms import axis_angle_to_rot6d
    norm = misc.Posenormalizer(None, device='cpu', normalize=True, min_max=False, rot_rep='rot6d')
    pose = synthetic.toy_poses()[:n].float()
    return norm.offline_normalize(axis_angle_to_rot6d(pose.reshape(-1, 3)).reshape(n, -1))


@pytest.mark.parametrize('method', ['RK45', 'RK23'])
def test_likelihood_vs_scipy_over_the_oracle(sd126, method):
    """get_likelihood_fn at 126 (RK45: the device integrator; RK23: scipy on the host over the native drift) on four rot6d
    poses with a fixed Rademacher probe, against scipy's solve_ivp over the oracle's drift and autograd divergence:
    bits/dim <= 2e-3, latent <= 5e-3, NFE within 25 %."""
    from scipy import integrate
    from oracle import score_ref as S
    B = 4
    data = _rot6d_poses(B)
    assert data.shape == (B, D)
    eps = torch.randint(0, 2, (B, D), generator=torch.Generator().manual_seed(11)).float() * 2 - 1
    osde = S.SubVP(0.1, 20., 1000)

    def rhs(t, y):
        x = torch.tensor(y[:-B], dtype=torch.float32).reshape(B, D).requires_grad_(True)
        tt = torch.full((B,), float(t))
        drift = S.reverse_drift(sd126, osde, x, tt, probability_flow=True)[0]
        div = (torch.autograd.grad((drift * eps).sum(), x)[0] * eps).sum(1)
        return np.concatenate([drift.detach().reshape(-1).numpy(), div.numpy()]).astype(np.float64)

    sol = integrate.solve_ivp(rhs, (1e-5, 1.0), np.concatenate([data.reshape(-1).numpy(), np.zeros(B)]), rtol=1e-5,
                              atol=1e-5, method=method)
    zr = torch.tensor(sol.y[:-B, -1], dtype=torch.float32).reshape(B, D)
    sde = sde_lib.subVPSDE(0.1, 20., 1000)
    bpd_ref = -(sde.prior_logp(zr) + torch.tensor(sol.y[-B:, -1], dtype=torch.float32)) / np.log(2) / D
    model = synthetic.make_score_model(42, pose_dim=6).cuda()
    fn = likelihood.get_likelihood_fn(sde, lambda v: v, rtol=1e-5, atol=1e-5, method=method, eps=1e-5)
    bpd, z, nfe = fn(model, data.cuda(), epsilon=eps.cuda())
    assert z.shape == (B, D) and bpd.shape == (B,)
    assert max_rel(bpd, bpd_ref) < 2e-3
    assert max_rel(z, zr) < 5e-3
    assert abs(nfe - sol.nfev) <= 0.25 * sol.nfev, (nfe, sol.nfev)


def test_ode_sampler_vs_oracle_rk45(sd126):
    """The device RK45 probability-flow ODE sampler at 126 on both engines against scipy RK45 over the oracle's drift."""
    from scipy import integrate
    from oracle import score_ref as S
    B = 16
    z0 = torch.randn(B, D, generator=torch.Generator().manual_seed(21))
    osde = S.SubVP(0.1, 20., 1000)

    def rhs(t, xf):
        x = torch.tensor(xf, dtype=torch.float32).reshape(B, D)
        return S.reverse_drift(sd126, osde, x, torch.ones(B) * float(t), probability_flow=True)[0].reshape(-1).numpy()

    sol = integrate.solve_ivp(rhs, (1.0, 1e-3), z0.reshape(-1).numpy(), rtol=1e-5, atol=1e-5, method='RK45')
    ref = torch.tensor(sol.y[:, -1], dtype=torch.float32).reshape(B, D)
    model = synthetic.make_score_model(42, pose_dim=6).cuda()
    fn = sampling.get_ode_sampler(sde_lib.subVPSDE(0.1, 20., 1000), (B, D), lambda x: x, eps=1e-3, device='cuda')
    for engine, tol in [(L.ENGINE_FP32, 2e-3), (L.ENGINE_TC, 5e-3)]:
        model.engine = engine
        nfe, x = fn(model, z=z0)
        assert x.shape == (B, D)
        assert rel_err(x, ref) < tol, (engine, float(rel_err(x, ref)))
        assert abs(nfe - sol.nfev) <= 0.25 * sol.nfev, (nfe, sol.nfev)
    model.engine = L.ENGINE_AUTO
