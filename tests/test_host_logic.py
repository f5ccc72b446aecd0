"""CPU: host-side logic of the product package (tables, masks, shards, drop-in surface) and the
C-ABI library: it must load and export every symbol include/dposer_b200.h declares.  No compute
call is made here (there is no CPU fallback to call)."""
import ctypes
import math
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, golden
from dposer_b200 import _lib as L
from dposer_b200 import misc, sde_lib, synthetic, utils as mutils
from oracle import score_ref as S


def test_library_loads_and_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, 'include', 'dposer_b200.h')).read()
    declared = sorted(set(re.findall(r'\b(dpb_[a-z0-9_]+)\s*\(', hdr)))
    assert len(declared) >= 20
    lib = L.load()
    for name in declared:
        assert hasattr(lib, name), f'{name} declared in include/dposer_b200.h but not exported'
    assert sorted(L.EXPORTS) == declared
    assert lib.dpb_version() == 100


def test_no_cpu_fallback_fails_loudly():
    m = synthetic.make_score_model()
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    with pytest.raises(RuntimeError):
        m(torch.zeros(2, 63), torch.ones(2))
    from dposer_b200.body_model import BodyModel
    bm = BodyModel(synthetic.make_body_tensors('smpl'), batch_size=2, model_type='smpl')
    with pytest.raises(RuntimeError):
        bm(pose_body=torch.zeros(2, 69))
    # the library itself reports the missing device instead of computing on the host
    sm = ctypes.c_int()
    assert L.load().dpb_device_info(0, ctypes.byref(sm), None, None) == L.ECUDA


def test_state_dict_surface_matches_reference_keys():
    m = synthetic.make_score_model()
    keys = set(m.state_dict().keys())
    expect = {'sigmas'}
    for n in ['pre_dense', 'pre_dense_t', 'pre_dense_cond', 'pre_gnorm', 'shared_time_embed.0', 'post_dense'] + \
             [f'b{b}_{k}' for b in (1, 2) for k in ('dense1', 'dense1_t', 'gnorm1', 'dense2', 'dense2_t', 'gnorm2')]:
        expect |= {n + '.weight', n + '.bias'}
    assert keys == expect
    assert sum(p.numel() for p in m.parameters()) == 8277567          # SURVEY Appendix D
    fp = golden('weights_fingerprint.npz')
    sd = m.state_dict()
    for k in fp.files:
        assert math.fsum(sd[k].double().abs().flatten().tolist()) == float(fp[k]), k


def test_em_coefficients_reproduce_the_reference_update(oracle_sd):
    """a*x + b*raw + c*z must equal EulerMaruyamaPredictor.update_fn on the oracle (fp32 rounding only)."""
    model = synthetic.make_score_model()
    g = torch.Generator().manual_seed(0)
    for N, pf in [(1000, False), (500, False), (1000, True)]:
        sde, osde = sde_lib.subVPSDE(0.1, 20., N), S.SubVP(0.1, 20., N)
        ts = mutils.timestep_grid(sde, 1e-3)
        coef, labels = mutils.em_coefficients(sde, model, ts, pf)
        assert np.array_equal(labels.long().numpy(), (ts * 999).long().numpy())
        for i in [0, N // 2, N - 1]:
            x = torch.randn(4, 63, generator=g)
            z = torch.randn(4, 63, generator=g)
            vt = torch.ones(4) * ts[i]
            raw = S.score_model_forward(oracle_sd, x, vt * 999, scale_by_sigma=False)
            xr, xmr = S.em_step(oracle_sd, osde, x, vt, z, pf)
            a, b, c = coef[i, 0], coef[i, 1], coef[i, 2]
            xm = a * x + b * raw
            assert (xm - xmr).abs().max() <= 2e-6 * xmr.abs().max()
            assert ((xm + c * z) - xr).abs().max() <= 2e-6 * xr.abs().max()
            mean, std = osde.marginal(torch.ones(1, 1), ts[i:i + 1])
            assert coef[i, 3] == mean[0, 0] and coef[i, 4] == std[0]


@pytest.mark.parametrize('sde_name,tag,pred', [('ve', 've_em', 'euler_maruyama'), ('ve', 've_rd', 'reverse_diffusion'),
                                               ('ve', 've_anc', 'ancestral_sampling'), ('vp', 'vp_rd', 'reverse_diffusion'),
                                               ('vp', 'vp_anc', 'ancestral_sampling'), ('sub', 'sub_rd', 'reverse_diffusion')])
def test_predictor_tables_reproduce_reference_chains(oracle_sd, sde_name, tag, pred):
    """The per-step (a, b, c) tables of every predictor / SDE pair, iterated on the CPU with the oracle's network output
    as ``raw``, land on the REAL reference's 8-step chains (sde_variants_golden.npz, replayed draws)."""
    g = golden('sde_variants_golden.npz')
    model = synthetic.make_score_model(42)
    if sde_name == 've':
        sde, eps, start, z0 = sde_lib.VESDE(0.01, 50., 8), 1e-5, 0, g['ve_em_z0']
    else:
        sde = sde_lib.VPSDE(0.1, 20., 1000) if sde_name == 'vp' else sde_lib.subVPSDE(0.1, 20., 1000)
        eps, start, z0 = 1e-3, 992, g['vp_em_z0']
    ts = mutils.timestep_grid(sde, eps)[start:]
    coef, labels = mutils.em_coefficients(sde, model, ts, False, True, predictor=pred)
    x = torch.tensor(z0)
    noise = torch.tensor(g[f'{tag}_noise'])
    for i in range(8):
        raw = S.score_model_forward(oracle_sd, x, torch.ones(x.shape[0]) * labels[i], scale_by_sigma=False)
        xm = coef[i, 0] * x + coef[i, 1] * raw
        x = xm + coef[i, 2] * noise[i]
    assert (xm - torch.tensor(g[f'{tag}_out'])).abs().max() <= 2e-4 * np.abs(g[f'{tag}_out']).max()
    assert (x - torch.tensor(g[f'{tag}_last'])).abs().max() <= 2e-4 * np.abs(g[f'{tag}_last']).max()


def test_prior_scalars_match_oracle():
    model = synthetic.make_score_model()
    sde, osde = sde_lib.subVPSDE(0.1, 20., 1000), S.SubVP()
    ts = mutils.timestep_grid(sde, 1e-3)
    for q in [0, 400, 799, 998]:
        ps = mutils.prior_scalars(sde, model, float(ts[q]))
        a, s = osde.alpha_sigma(ts[q:q + 1])
        assert ps['alpha'] == float(a[0, 0]) and ps['std'] == float(s[0])
        sig = S.sigma_table()[(ts[q] * 999).long()]
        np.testing.assert_allclose(ps['inv_sigma_std'], float(1 / (sig * s[0])), rtol=1e-6)


def test_masks_parts_shards_schedules_bit_exact():
    g = golden('int_tables.npz')
    for part in ['legs', 'arms', 'trunk', 'hands', 'left_leg', 'right_leg', 'left_arm', 'right_arm']:
        assert getattr(misc.BodyPartIndices, part) == g[f'part_{part}'].tolist()
        mask, obs = misc.create_mask(torch.zeros(3, 63), part=part)
        assert np.array_equal(np.nonzero(mask[0].numpy() == 0)[0], g[f'maskzero_{part}'])
        assert (obs[:, mask[0] == 1] == 0).all()
    for N, total, trun, off, nm in [(1000, 200, 5.0, 2, 'completion'), (500, 180, 4.0, 2, 'denoise'),
                                    (500, 500, 20.0, 5, 'smplify')]:
        assert misc.quan_t_schedule(N, total, trun, off) == g[f'quan_t_{nm}'].tolist()
    for total, world, r, first, n in g['shards'].tolist():
        st, cnt = misc.shard_range(total, world, r)
        assert cnt == n and (n == 0 or st == first)
    # shards tile the range exactly, in rank order
    for total, world in [(500, 8), (65536, 8), (40960, 3), (5, 8)]:
        pos = 0
        for r in range(world):
            st, cnt = misc.shard_range(total, world, r)
            assert st == pos
            pos += cnt
        assert pos == total


def test_create_mask_same_draws_as_reference_rng():
    """With the same torch seed the noise fill equals the reference's (same randn_like call order)."""
    g = golden('sampler_golden.npz')
    norm = misc.Posenormalizer(None, device='cpu', normalize=True, min_max=False, rot_rep='axis')
    poses = norm.offline_normalize(synthetic.toy_poses()[:5])
    torch.manual_seed(3)
    mask, obs = misc.create_mask(poses, part='legs')
    assert np.array_equal(mask.numpy(), g['comp8_mask']) and np.array_equal(obs.numpy(), g['comp8_obs'])


def test_normalizer_roundtrip_and_stats():
    norm = misc.Posenormalizer(None, device='cpu', normalize=True, min_max=False, rot_rep='axis')
    toy = synthetic.toy_poses()
    x = norm.offline_normalize(toy)
    assert (norm.offline_denormalize(x) - toy).abs().max() < 1e-6
    g = golden('score_golden.npz')
    gen = torch.Generator().manual_seed(5)
    x7 = norm.offline_normalize(toy[:7]) + 0.3 * torch.randn(7, 63, generator=gen)
    assert np.array_equal(x7.numpy(), g['x'])


def test_normalizer_rot6d_and_mean_pose_observation():
    """Posenormalizer(rot_rep='rot6d') (AMASS.py:187-259 with the reference's own rot6d statistics) and create_mask's
    mean-pose observation (misc.py:43-53).  The rot6d conversion itself is the restated torchgeometry path (unpinned)."""
    from dposer_b200 import transforms as T
    toy = synthetic.toy_poses()[:64]
    for min_max in (False, True):
        norm = misc.Posenormalizer(None, device='cpu', normalize=True, min_max=min_max, rot_rep='rot6d')
        assert norm.mean_poses.shape == (126,) and norm.min_poses.shape == (126,)
        x = norm.offline_normalize(toy, from_axis=True)
        assert x.shape == (64, 126) and torch.isfinite(x).all()
        r6 = T.axis_angle_to_rot6d(toy.reshape(-1, 3)).reshape(64, 126)
        ref = (2 * (r6 - norm.min_poses) / (norm.max_poses - norm.min_poses) - 1) if min_max else \
            (r6 - norm.mean_poses) / norm.std_poses
        assert torch.equal(x, ref)
        assert (norm.offline_denormalize(x) - r6).abs().max() < 1e-5
        back = norm.offline_denormalize(x, to_axis=True)
        assert (back - toy).abs().max() < 5e-4                # fp32 round trip; AMASS body poses are far from the pi branch
        x3 = norm.offline_normalize(toy[None].repeat(2, 1, 1), from_axis=True)      # [t, b, dim]
        assert torch.equal(x3[1], x)
    # AMASS-like data should look standardised under the reference's mean / std
    norm = misc.Posenormalizer(None, device='cpu', normalize=True, min_max=False, rot_rep='rot6d')
    z = norm.offline_normalize(synthetic.toy_poses(), from_axis=True)
    assert float(z.mean().abs()) < 0.5 and 0.3 < float(z.std()) < 3.0
    # mean-pose observation: masked joints carry the SMPL mean pose, the rest is untouched
    mean6 = torch.tensor(np.load(os.path.join(os.path.dirname(synthetic.__file__), 'data', 'smpl_mean_params.npz'))['pose'][6:])
    for rot_n, data in ((3, toy), (6, r6)):
        mask, obs = misc.create_mask(data, part='left_arm', observation_type='mean')
        keep = mask.bool()
        assert torch.equal(obs[keep], data[keep])
        idx = (~keep[0]).nonzero().flatten()
        fill = mean6.float() if rot_n == 6 else T.rot6d_to_axis_angle(mean6.float().reshape(-1, 6)).reshape(-1)
        assert torch.equal(obs[:, idx], fill[idx][None].repeat(64, 1))


def test_sde_objects_match_oracle_scalars():
    sde, osde = sde_lib.subVPSDE(0.1, 20., 1000), S.SubVP()
    t = torch.linspace(1, 1e-3, 1000)
    x = torch.randn(1000, 3)
    assert torch.equal(sde.sde(x, t)[1], osde.sde(x, t)[1])
    assert torch.equal(sde.marginal_prob(x, t)[1], osde.marginal(x, t)[1])
    assert torch.equal(sde.return_alpha_sigma(t)[0], osde.alpha_sigma(t)[0])
    k = golden('known_answers.npz')
    assert np.array_equal(sde.alphas.numpy(), k['sde_alphas'])
    with pytest.raises(NotImplementedError):
        mutils.get_score_fn(object(), None)
    # reverse() keeps the reference surface
    r = sde.reverse(lambda x, t, c, m: torch.zeros_like(x), probability_flow=True)
    d, g_ = r.sde(x[:4], t[:4])
    assert d.shape == (4, 3) and float(g_) == 0.0 and r.N == 1000 and r.T == 1


def test_sampling_fn_argument_errors():
    from dposer_b200 import sampling
    cfg = synthetic.default_config()
    cfg.sampling.method = 'bogus'
    with pytest.raises(ValueError):
        sampling.get_sampling_fn(cfg, sde_lib.subVPSDE(), (2, 63), lambda x: x, 1e-3, device='cpu')
    cfg.sampling.method = 'pc'
    cfg.sampling.predictor = 'ancestral_sampling'
    with pytest.raises(NotImplementedError):
        sampling.get_sampling_fn(cfg, sde_lib.subVPSDE(), (2, 63), lambda x: x, 1e-3, device='cpu')


def test_body_model_wrapper_shapes_and_joint_map():
    from dposer_b200 import body_model as bmod
    g = golden('int_tables.npz')
    assert bmod.JOINT_MAP_49 == g['smplx_joint_map49'].tolist()
    assert bmod.SMPLX_PARENTS[:22] == bmod.SMPL_PARENTS[:22] and len(bmod.SMPLX_PARENTS) == 55
    # first 22 parents are what lib/body_model/utils.py:180-205 (get_smpl_skeleton) implies
    assert bmod.SMPL_PARENTS[:22] == [-1, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19]
    with pytest.raises(ValueError):
        bmod.BodyModel(synthetic.make_body_tensors('smpl'), model_type='smplx')
    m = bmod.SMPLX(synthetic.make_body_tensors('smplx'))
    assert m.mean_poses.shape == (72,) and m.mean_shape.shape == (10,)
    assert torch.isfinite(m.mean_poses).all()


def test_rot6d_transforms_properties():
    """lib/utils/transforms.py:197-255 restated without torchgeometry (parity unpinned): round trips, orthonormality and
    agreement with the LBS oracle's Rodrigues formula."""
    from dposer_b200 import transforms as T
    from oracle import lbs_ref
    g = torch.Generator().manual_seed(5)
    aa = torch.randn(200, 3, generator=g) * 1.2
    aa[0] = 0.
    aa[1] = torch.tensor([1e-8, 0., 0.])
    aa[2] = torch.tensor([3.1, 0.1, -0.05])          # close to pi
    R = T.axis_angle_to_mat3x3(aa)
    assert float((R @ R.transpose(1, 2) - torch.eye(3)).abs().max()) < 1e-5
    assert float((torch.linalg.det(R) - 1).abs().max()) < 1e-5
    assert float((R[3:] - lbs_ref.batch_rodrigues(aa[3:])).abs().max()) < 1e-5
    r6 = T.axis_angle_to_rot6d(aa)
    assert r6.shape == (200, 6)
    assert float((T.rot6d_to_mat3x3(r6) - R).abs().max()) < 1e-5
    back = T.rot6d_to_axis_angle(r6)
    assert float((T.axis_angle_to_mat3x3(back) - R).abs().max()) < 2e-5      # same rotation (axis-angle is 2-to-1 at pi)
    small = aa.norm(dim=1) < 3.0
    assert float((back[small] - aa[small]).abs().max()) < 2e-5


def test_rot6d_gram_schmidt_vs_reference_golden():
    """lib/utils/transforms.py:225-234 (`rot6d_to_mat3x3`, pure torch in the reference): bit-exact against the fixture the
    real reference wrote (tests/golden/make_rot6d_golden.py), including non-orthonormal, tiny and huge inputs."""
    from dposer_b200 import transforms as T
    gd = golden('rot6d_golden.npz')
    R = T.rot6d_to_mat3x3(torch.from_numpy(gd['rot6d']))
    assert torch.equal(R, torch.from_numpy(gd['mat']))
    # the axis-angle leg (torchgeometry in the reference: unpinned) must at least describe the same rotation
    aa = T.rot6d_to_axis_angle(torch.from_numpy(gd['rot6d']))
    assert float((T.axis_angle_to_mat3x3(aa) - R).abs().max()) < 2e-5


def test_rot6d_helpers_vs_torchgeometry_restatement():
    """The legs of lib/utils/transforms.py:197-258 that call torchgeometry (absent; oracle/tgm_ref.py restates its published
    0.1.2 algorithms, parity unpinned): the product helpers agree with them to fp32 rounding.  torchgeometry's axis is
    `aa / (theta + 1e-6)` -- a relative 1e-6 / theta shortening the product does not reproduce: tolerance 4e-6 on matrix
    entries.  Small components must survive the matrix -> axis-angle leg (a sqrt(1 +- Rii)-only extraction loses ~3e-4)."""
    from dposer_b200 import transforms as T
    from oracle import tgm_ref as G
    g = torch.Generator().manual_seed(5)
    aa = torch.randn(4000, 3, generator=g) * 1.2
    aa[0] = 0.
    aa[1] = torch.tensor([1e-8, 0., 0.])
    aa[2] = torch.tensor([3.1, 0.1, -0.05])
    aa[3] = torch.tensor([5e-4, 5e-4, 5e-4])                      # below torchgeometry's Taylor threshold (theta^2 <= 1e-6)
    aa[4] = torch.tensor([1.0923, 1.3298, -2.98e-4])              # one tiny component
    aa[5] = torch.tensor([0., -3.1415, 1e-3])                     # next to pi
    assert float((T.axis_angle_to_mat3x3(aa) - G.axis_angle_to_mat3x3(aa)).abs().max()) < 4e-6
    assert float((T.axis_angle_to_rot6d(aa) - G.axis_angle_to_rot6d(aa)).abs().max()) < 4e-6
    r6 = T.axis_angle_to_rot6d(aa)
    ours, ref = T.rot6d_to_axis_angle(r6.clone()), G.rot6d_to_axis_angle(r6.clone())
    below_pi = aa.norm(dim=1) < 3.0                               # at pi the two sign conventions may differ
    assert float((ours - ref)[below_pi].abs().max()) < 5e-6
    assert float((ours - aa)[below_pi].abs().max()) < 5e-6        # incl. the -2.98e-4 component of row 4
    R = T.axis_angle_to_mat3x3(aa)
    assert float((T.axis_angle_to_mat3x3(ours) - R).abs().max()) < 5e-6
    assert float((T.axis_angle_to_mat3x3(ref) - R).abs().max()) < 5e-6
    deg = torch.zeros(2, 6)                                       # degenerate input: NaN -> 0 like the reference
    assert torch.equal(T.rot6d_to_axis_angle(deg), torch.zeros(2, 3))


def test_rk45_controller_reproduces_scipy_solve_ivp():
    """dposer_b200.ode: the host-side step-size controller (scipy's RungeKutta._step_impl / select_initial_step restated)
    over a numpy stand-in for the native stage / error kernels lands on solve_ivp(method='RK45') itself: same number of
    function evaluations, same final state; and the Butcher tableau the kernels carry equals scipy's."""
    import re
    from scipy import integrate
    from dposer_b200 import ode
    RK = integrate.RK45
    src = open(os.path.join(ROOT, 'dposer_b200', 'csrc', 'rk45.cu')).read()

    def table(name):
        body = re.search(name + r'\[[^\]]*\](?:\[[^\]]*\])?\s*=\s*\{(.*?)\};', src, re.S).group(1)
        return [eval(x.replace('.0', '.0')) for x in re.sub(r'[{}\s]', '', body).split(',') if x]
    A = np.array(table('A')).reshape(6, 5)
    assert np.allclose(A, RK.A, rtol=0, atol=1e-16) and np.allclose(table('Bc'), RK.B, atol=1e-16)
    assert np.allclose(table('Ec'), RK.E, atol=1e-16) and np.allclose(ode.C_NODES, RK.C, atol=1e-16)

    class NumpyBackend(ode.Backend):
        def __init__(self, fun, y0):
            self.fun, self.y, self.n = fun, np.array(y0, float), len(y0)
            self.k = np.zeros((7, self.n))

        def eval_initial(self, t):
            self.k[0] = self.fun(t, self.y)

        def eval_stage(self, s, t, h):
            self.k[s] = self.fun(t, self.y + np.dot(self.k[:s].T, RK.A[s, :s]) * h)

        def eval_candidate(self, t, h):
            self.y_new = self.y + h * np.dot(self.k[:-1].T, RK.B)
            self.k[6] = self.fun(t, self.y_new)

        def error_norm(self, h, rtol, atol):
            scale = atol + np.maximum(np.abs(self.y), np.abs(self.y_new)) * rtol
            e = np.dot(self.k.T, RK.E) * h / scale
            return np.linalg.norm(e) / e.size ** 0.5

        def accept(self):
            self.y, self.k[0] = self.y_new, self.k[6]

        def initial_step_norms(self, t0, direction, rtol, atol, interval):
            return ode.select_initial_step(self.y, self.k[0].copy(), self.fun, t0, direction, rtol, atol, interval)

    W = np.random.default_rng(0).standard_normal((12, 12)) * 0.7

    def fun(t, y):                                  # stiff-ish nonlinear system, time dependent
        return np.tanh(W @ y) * (1 + 3 * t) - 0.5 * y + np.sin(5 * t)
    y0 = np.linspace(-1, 1, 12)
    for (t0, t1, rtol, atol) in [(1e-5, 1.0, 1e-5, 1e-5), (1.0, 1e-3, 1e-5, 1e-5), (0.0, 2.0, 1e-3, 1e-6)]:
        ref = integrate.solve_ivp(fun, (t0, t1), y0, rtol=rtol, atol=atol, method='RK45')
        be = NumpyBackend(fun, y0)
        nfev, attempts = ode.solve_rk45(be, t0, t1, rtol=rtol, atol=atol)
        assert nfev == ref.nfev, (nfev, ref.nfev)
        assert np.abs(be.y - ref.y[:, -1]).max() <= 1e-12 * max(1.0, np.abs(ref.y[:, -1]).max())


def test_training_host_surface_without_a_gpu():
    """losses / ema on the host: no CPU fallback (loudly), argument errors, the EMA decay schedule and Adam's scalars."""
    from dposer_b200 import ema as ema_mod
    from dposer_b200 import losses
    cfg = synthetic.default_config()
    model = synthetic.make_score_model(42)                     # CPU parameters
    with pytest.raises(RuntimeError):
        losses.get_optimizer(cfg, model.parameters())          # flat buffers live on the device
    sde = sde_lib.subVPSDE(0.1, 20., 1000)
    with pytest.raises(NotImplementedError):
        losses.get_sde_loss_fn(sde, True, return_data=True)
    with pytest.raises(ValueError):
        losses.get_step_fn(sde_lib.subVPSDE(0.1, 20., 1000), True, continuous=False)      # discrete training: VE / VP only
    with pytest.raises(NotImplementedError):
        losses.get_step_fn(sde, True, auxiliary_loss=True, denormalize=lambda v: v, body_model=object(), rot_rep='rot6d')
    fn = losses.get_sde_loss_fn(sde, True, reduce_mean=True)
    with pytest.raises(RuntimeError):
        fn(model, torch.zeros(4, 63), None, None)              # batch on the CPU
    # per-row scalars of the three loss families (host fp32, the reference's expressions)
    t = torch.tensor([0.25, 0.5, 1.0])
    rows = fn.make_rows(model, 3, t)
    mean, std = sde.marginal_prob(torch.ones(3, 1), t)
    assert rows.shape == (6, 3) and torch.equal(rows[0], t * 999) and torch.equal(rows[1], mean[:, 0]) and torch.equal(rows[2], std)
    sig = mutils.sigma_at(model, t * 999)
    assert torch.allclose(rows[3], -1.0 / sig, rtol=1e-6) and torch.equal(rows[4], torch.ones(3))        # e = -res / sigma + z
    assert torch.allclose(rows[5], torch.full((3,), 1.0 / 63))
    lw = losses.get_sde_loss_fn(sde, True, reduce_mean=False, likelihood_weighting=True).make_rows(model, 3, t)
    g2 = sde.sde(torch.zeros(3, 1), t)[1] ** 2
    assert torch.allclose(lw[5], 0.5 * g2) and torch.allclose(lw[4], 1.0 / std)
    with pytest.raises(ValueError):
        ema_mod.ExponentialMovingAverage(model.parameters(), decay=1.5)
    e = ema_mod.ExponentialMovingAverage(model.parameters(), decay=0.9999)
    seq = []
    for n in range(1, 6):
        seq.append(e.next_one_minus_decay())
        e.num_updates += 1
    assert np.allclose(seq, [1 - min(0.9999, (1 + n) / (10 + n)) for n in range(1, 6)])
    sd = e.state_dict()
    assert set(sd) == {'decay', 'num_updates', 'shadow_params'} and len(sd['shadow_params']) == len(list(model.parameters()))


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the driver's CPU arm): rank 0 prints ONE JSON line with the contract's keys, the
    cpu_baseline that describes the run and a zero-copy e2e equal to the line's own value; other ranks print nothing and
    exit 0.  On this container oracle/_ref is staged by build(), so the arm is the reference's own sampler."""
    import json
    import subprocess
    import sys
    env = dict(os.environ, RANK='1', WORLD_SIZE='2', LOCAL_RANK='1')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--steps', '1',
                        '--warmup', '1'], env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ''
    env = {k: v for k, v in os.environ.items() if k not in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK')}
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '1', '--steps', '1',
                        '--warmup', '1'], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-800:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
              'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert k in d, k
    assert d['impl'] == 'reference' and d['unit'] == 'poses/s' and d['higher_is_better'] is True and d['vs_baseline'] is None
    assert d['metric'].startswith('poses/sec') and 'workload' in d['config'] and 'model' not in d['config']
    cb = d['cpu_baseline']
    assert cb['value'] == d['value'] > 0 and cb['cores'] >= 1 and cb['kind'] in ('reference', 'port') and cb['sample']
    if os.path.isdir(os.path.join(ROOT, 'oracle', '_ref', 'lib')):
        assert cb['kind'] == 'reference'
    assert d['e2e'] == {'value': d['value'], 'unit': 'poses/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
