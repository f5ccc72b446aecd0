"""CPU: the oracle must reproduce every golden vector produced by the REAL reference
(tests/golden/make_golden.py).  This is what pins the oracle (prompt section 3)."""
import math
import os

import numpy as np
import torch

from conftest import golden
from oracle import fitting_ref as Fr
from oracle import score_ref as S


def test_known_answers_appendix_d():
    k = golden('known_answers.npz')
    sde = S.SubVP(0.1, 20., 1000)
    ts = torch.linspace(1, 1e-3, 1000)
    t5 = ts[torch.tensor(k['i'])]
    assert np.array_equal(t5.numpy(), k['t'])
    assert np.array_equal((t5 * 999).long().numpy(), k['idx'])
    assert np.array_equal(sde.sde(torch.zeros(5, 1), t5)[1].numpy(), k['g'])
    assert np.array_equal(sde.alpha_sigma(t5)[1].numpy(), k['std'])
    assert np.array_equal(S.sigma_table()[k['idx']].numpy(), k['sigmas'])
    assert np.array_equal(S.timestep_embedding(torch.tensor([499.5]))[0].numpy(), k['temb_4995'])
    assert np.array_equal(sde.alphas.numpy(), k['sde_alphas'])
    assert np.array_equal((ts * 999).long().numpy(), k['all_idx'])
    # SURVEY Appendix D printed values
    assert k['idx'].tolist() == [999, 500, 499, 1, 0]
    np.testing.assert_allclose(k['g'][0], 4.472136021, rtol=1e-7)
    np.testing.assert_allclose(k['std'][4], 1.099705696e-04, rtol=1e-6)


def test_weight_recipe_fingerprint(oracle_sd):
    fp = golden('weights_fingerprint.npz')
    for k in fp.files:
        assert math.fsum(oracle_sd[k].double().abs().flatten().tolist()) == float(fp[k]), k


def test_score_net_matches_reference(oracle_sd):
    g = golden('score_golden.npz')
    x = torch.tensor(g['x'])
    sde = S.SubVP()
    for tv in ['1.0', '0.5', '0.1', '0.01', '0.001']:
        vt = torch.ones(7) * float(tv)
        assert np.array_equal(S.score_fn(oracle_sd, sde, x, vt).numpy(), g[f'score_{tv}'])
        assert np.array_equal(S.score_model_forward(oracle_sd, x, vt * 999).numpy(), g[f'model_{tv}'])
    vt = torch.tensor(g['t_mixed'])
    assert np.array_equal(S.score_model_forward(oracle_sd, x, vt * 999).numpy(), g['model_mixed'])


def _noise_dict(g, name, start):
    n = g[f'{name}_noise_pred'].shape[0]
    out = {}
    for i in range(n):
        d = {'pred': torch.tensor(g[f'{name}_noise_pred'][i])}
        for k in ('corr', 'imp_c', 'imp_p'):
            if f'{name}_noise_{k}' in g.files:
                d[k] = torch.tensor(g[f'{name}_noise_{k}'][i])
        out[start + i] = d
    return out


def test_pc_sampler_matches_reference(oracle_sd):
    g = golden('sampler_golden.npz')
    cases = [('em8', 8, 'none', None, False, 0), ('em32', 32, 'none', None, False, 0),
             ('lang8', 1000, 'langevin', 'denoise', False, 992), ('comp8', 8, 'none', 'completion', False, 0),
             ('ode8', 8, 'none', None, True, 0), ('den16', 16, 'none', 'denoise', False, 10)]
    for name, N, corr, task, pf, start in cases:
        obs = torch.tensor(g[f'{name}_obs']) if f'{name}_obs' in g.files else None
        mask = torch.tensor(g[f'{name}_mask']) if f'{name}_mask' in g.files else None
        traj, out = S.pc_sample(oracle_sd, S.SubVP(0.1, 20., N), torch.tensor(g[f'{name}_z0']), 1e-3,
                                noise=_noise_dict(g, name, start), corrector=corr, observation=obs, mask=mask,
                                task=task, start_step=start, probability_flow=pf, keep_traj=True)
        assert np.array_equal(out.numpy(), g[f'{name}_out']), name
        assert np.array_equal(traj[-1].numpy(), g[f'{name}_traj_last']), name


def test_prior_loss_matches_reference(oracle_sd):
    g = golden('prior_golden.npz')
    x0 = torch.tensor(g['x0'])
    sde = S.SubVP()
    ts = torch.linspace(1, 1e-3, 1000)
    for name, qt in [('q799', 799), ('q998', 998), ('q400', 400)]:
        l, gr = S.prior_loss(oracle_sd, sde, x0, torch.ones(7) * ts[qt], torch.tensor(g[f'{name}_z']), True, 'mean')
        assert np.array_equal(l.numpy(), g[f'{name}_loss']) and np.array_equal(gr.numpy(), g[f'{name}_grad'])
    for name, weighted, multi in [('md_plain', False, False), ('md_weighted', True, False), ('md_ddim', False, True)]:
        l, gr = S.prior_loss(oracle_sd, sde, x0, torch.ones(7) * ts[450], torch.tensor(g[f'{name}_z']), weighted,
                             'sum', divisor=7, multi_denoise=multi)
        assert np.array_equal(l.numpy(), g[f'{name}_loss']) and np.array_equal(gr.numpy(), g[f'{name}_grad'])


def test_integer_tables_bit_exact():
    g = golden('int_tables.npz')
    for part in ['legs', 'arms', 'trunk', 'hands', 'left_leg', 'right_leg', 'left_arm', 'right_arm']:
        assert Fr.BODY_PARTS[part] == g[f'part_{part}'].tolist()
        assert np.array_equal(np.sort(Fr.mask_indices(part).numpy()), g[f'maskzero_{part}'])
    assert g['maskzero_legs'].tolist() == [0, 1, 2, 3, 4, 5, 9, 10, 11, 12, 13, 14, 18, 19, 20, 21, 22, 23, 27, 28,
                                           29, 30, 31, 32]
    for N, total, trun, off, nm in [(1000, 200, 5.0, 2, 'completion'), (500, 180, 4.0, 2, 'denoise'),
                                    (500, 500, 20.0, 5, 'smplify')]:
        assert S.quan_t_schedule(N, total, trun, off) == g[f'quan_t_{nm}'].tolist()
    for total, world, r, first, n in g['shards'].tolist():
        st, cnt = Fr.shard_range(total, world, r)
        assert cnt == n and (n == 0 or st == first)


def test_fitting_losses_and_metrics_match_reference():
    g = golden('fitting_golden.npz')
    t = lambda k: torch.tensor(g[k])         # noqa: E731
    ints = golden('int_tables.npz')
    center = torch.full((6, 2), 512.)
    body = Fr.body_fitting_loss(t('pose'), t('betas'), t('joints'), center, t('kp'), t('conf'), t('prior'))
    cam = Fr.camera_fitting_loss(t('joints'), t('cam_t'), t('cam_est'), center, t('kp'), t('conf'),
                                 op_ind=ints['op_ind'], gt_ind=ints['gt_ind'])
    np.testing.assert_allclose(body.numpy(), g['body_loss'], rtol=1e-6)
    np.testing.assert_allclose(cam.numpy(), g['cam_loss'], rtol=1e-6)
    np.testing.assert_allclose(Fr.gaussian_smoothing(t('smooth_in'), 3, 2).numpy(), g['smooth_out'], rtol=1e-6,
                               atol=1e-7)
    a = golden('apd_golden.npz')
    np.testing.assert_allclose(Fr.apd(torch.tensor(a['joints'])).numpy(), a['apd'], rtol=1e-6)


def test_lbs_oracle_invariants():
    """LBS parity is unpinned (smplx absent); check the invariants any correct LBS satisfies."""
    from dposer_b200 import synthetic
    from oracle import lbs_ref
    m = synthetic.make_body_tensors('smpl')
    B = 3
    g = torch.Generator().manual_seed(0)
    betas = torch.randn(B, 10, generator=g)
    # zero pose: vertices equal the shaped template, joints equal the regressed rest joints
    v, j = lbs_ref.body_forward(m, betas, torch.zeros(B, 72))
    v_shaped = m['v_template'][None] + torch.einsum('bl,mkl->bmk', betas, m['shapedirs'])
    assert (v - v_shaped).abs().max() < 1e-6
    jrest = torch.einsum('bik,ji->bjk', v_shaped, m['J_regressor'])
    assert (j[:, :24] - jrest).abs().max() < 1e-6
    # root-only rotation: rigid motion about the pelvis rest joint
    pose = torch.zeros(B, 72)
    pose[:, :3] = torch.randn(B, 3, generator=g)
    v2, _ = lbs_ref.body_forward(m, betas, pose)
    R = lbs_ref.batch_rodrigues(pose[:, :3])
    expect = torch.einsum('bij,bvj->bvi', R, v_shaped - jrest[:, :1]) + jrest[:, :1]
    assert (v2 - expect).abs().max() < 2e-6
    assert j.shape == (B, 45, 3)


def test_task_loops_match_reference(oracle_sd):
    """oracle/fitting_loops.py against the REAL DPoserComp.optimize / MotionDenoise.optimize / SMPLify.__call__
    (tests/golden/make_golden_loops.py; reference draws replayed)."""
    from conftest import rel_err
    from dposer_b200 import synthetic
    from dposer_b200.body_model import JOINT_MAP_49
    from oracle import fitting_loops
    g = golden('loops_golden.npz')
    t = lambda k: torch.tensor(g[k])         # noqa: E731
    stats = np.load(os.path.join(os.path.dirname(synthetic.__file__), 'data', 'amass_stats.npz'))
    mean, std = torch.tensor(stats['mean_poses']), torch.tensor(stats['std_poses'])
    # completion
    iters, spi = g['comp_iters'].tolist()
    obs = t('comp_obs')
    out = fitting_loops.completion_optimize(oracle_sd, obs, t('comp_mask'), list(t('comp_z')), iterations=iters,
                                            steps_per_iter=spi)
    assert rel_err(out - obs, t('comp_out') - obs) < 1e-5
    # motion denoising: two sequences in one batch == two separate reference runs
    m = synthetic.make_body_tensors('smplx')
    seq_len, n_seq, iters, spi = g['md_geom'].tolist()
    init = t('md_init')
    pose = fitting_loops.motion_denoise(oracle_sd, m, t('md_noisy'), init, mean, std, list(t('md_z')), seq_len,
                                        sde_N=500, iterations=iters, steps_per_iter=spi, sample_trun=4.0)
    assert rel_err(pose - init, t('md_final') - init) < 2e-4
    # SMPLify: three images in one batch == three B=1 reference runs; hands at the model's non-zero mean pose
    (iters,) = g['sf_iters'].tolist()
    ip, ib, ic = t('sf_init_pose'), t('sf_init_betas'), t('sf_init_cam')
    pose, betas, cam = fitting_loops.smplify(oracle_sd, m, torch.tensor(JOINT_MAP_49), ip, ib, ic, t('sf_center'),
                                             t('sf_kp2d'), mean, std, list(t('sf_z')), num_iters=iters, sde_N=500,
                                             hand_mean=m['hands_mean'])
    assert rel_err(pose - ip, t('sf_pose') - ip) < 2e-4
    assert rel_err(betas - ib, t('sf_betas') - ib) < 2e-4
    assert rel_err(cam - ic, t('sf_cam') - ic) < 2e-4
    # the hand pose matters: with flat hands the same loop lands elsewhere (guards the SMPLX default semantics)
    pose0, _, _ = fitting_loops.smplify(oracle_sd, m, torch.tensor(JOINT_MAP_49), ip, ib, ic, t('sf_center'),
                                        t('sf_kp2d'), mean, std, list(t('sf_z')), num_iters=iters, sde_N=500)
    assert rel_err(pose0 - ip, t('sf_pose') - ip) > 1e-3


def test_lbs_two_independent_restatements_agree():
    """LBS parity is unpinned (smplx absent).  The torch-fp32 restatement (smplx structure: 4x4 matrices) and an
    independent float64 formulation (world rotations + posed joints, no homogeneous matrices) must agree to fp32
    round-off on SMPL and SMPL-X with every input exercised (hands, jaw, eyes, expression, translation)."""
    from dposer_b200 import synthetic
    from oracle import lbs_np64, lbs_ref
    for mt, tol in [('smpl', 2e-6), ('smplx', 2e-6)]:
        m = synthetic.make_body_tensors(mt)
        B = 4
        g = torch.Generator().manual_seed(5)
        J = m['J_regressor'].shape[0]
        pose = 0.4 * torch.randn(B, J * 3, generator=g)
        shape = torch.randn(B, m['shapedirs'].shape[2], generator=g)
        tr = torch.randn(B, 3, generator=g)
        v, j = lbs_ref.body_forward(m, shape, pose, tr)
        v64, j64 = lbs_np64.body_forward(m, shape, pose, tr)
        assert np.abs(v.numpy() - v64).max() < tol and np.abs(j.numpy() - j64).max() < tol
        assert j.shape[1] == J + 21 + (51 if mt == 'smplx' else 0)
        # invariants on BOTH: translation equivariance; a single non-root joint rotation leaves every vertex that
        # has no weight on that joint's subtree untouched
        v0, _ = lbs_np64.body_forward(m, shape, pose)
        assert np.abs(v64 - (v0 + tr.numpy()[:, None])).max() < 1e-12
        pose1 = torch.zeros(B, J * 3)
        jj = 18                                                  # left elbow: subtree = {18, 20, (hand joints)}
        pose1[:, jj * 3:jj * 3 + 3] = torch.randn(B, 3, generator=g)
        parents = m['parents']
        sub = {jj}
        for k in range(jj + 1, J):
            if parents[k] in sub:
                sub.add(k)
        untouched = (m['lbs_weights'][:, sorted(sub)].sum(1) == 0).numpy()
        zero = torch.zeros(B, J * 3)
        for fwd in (lambda p: lbs_ref.body_forward(m, shape, p)[0].numpy(),
                    lambda p: lbs_np64.body_forward(m, shape, p)[0]):
            a, b = fwd(pose1), fwd(zero)
            # posedirs move every vertex by the (R-I) feature of joint jj: remove that linear term first
            feat = (lbs_ref.batch_rodrigues(pose1[:, jj * 3:jj * 3 + 3]) - torch.eye(3)).reshape(B, 9).numpy()
            off = (feat @ m['posedirs'][(jj - 1) * 9:jj * 9].numpy().astype(np.float64)).reshape(B, -1, 3)
            assert np.abs((a - off)[:, untouched] - b[:, untouched]).max() < 2e-6
            assert np.abs(a[:, ~untouched] - b[:, ~untouched]).max() > 1e-3


def test_load_body_tensors_smplx_layout(tmp_path):
    """load_body_tensors on a file written in the smplx .npz layout (posedirs [V,3,P], shapedirs with 300 shape +
    expression components, kintree_table, f, weights, lmk_*, hands_mean*) gives back the tensors LbsCore expects."""
    from dposer_b200 import synthetic
    from dposer_b200.body_model import load_body_tensors
    m = synthetic.make_body_tensors('smplx')
    V, J = 10475, 55
    sd = np.zeros((V, 3, 310), np.float32)
    sd[:, :, :10] = m['shapedirs'][:, :, :10].numpy()
    sd[:, :, 300:310] = m['shapedirs'][:, :, 10:].numpy()
    faces = m['faces'].numpy()
    lmk_idx = np.arange(51) * 7
    faces[lmk_idx] = m['lmk_faces'].numpy()
    kt = np.stack([np.array([2 ** 32 - 1] + m['parents'][1:], np.int64), np.arange(J)])
    path = str(tmp_path / 'SMPLX_SYNTH.npz')
    np.savez(path, v_template=m['v_template'].numpy(), shapedirs=sd,
             posedirs=m['posedirs'].numpy().T.reshape(V, 3, -1), J_regressor=m['J_regressor'].numpy(),
             weights=m['lbs_weights'].numpy(), kintree_table=kt, f=faces, lmk_faces_idx=lmk_idx,
             lmk_bary_coords=m['lmk_bary'].numpy(), hands_meanl=m['hands_mean'][:45].numpy(),
             hands_meanr=m['hands_mean'][45:].numpy())
    t = load_body_tensors(path, 'smplx')
    for k in ['v_template', 'shapedirs', 'posedirs', 'J_regressor', 'lbs_weights', 'lmk_bary', 'hands_mean']:
        assert torch.equal(t[k], m[k]), k
    assert t['parents'] == m['parents'] and torch.equal(t['lmk_faces'], m['lmk_faces'])


def test_training_oracle_reproduces_reference_steps():
    """oracle/train_ref.py against the REAL reference's three training steps (train_golden.npz): loss, gradient norm and
    sampled gradients per step, sampled parameter / EMA deltas at the end."""
    from oracle import score_ref as S
    from oracle import train_ref as T
    g = golden('train_golden.npz')
    B, STEPS = 96, 3
    sd = S.make_state_dict(42)
    names = T.param_names(sd)
    sd0 = {k: sd[k].clone() for k in names}
    opt = {k: (torch.zeros_like(sd[k]), torch.zeros_like(sd[k])) for k in names}
    opt['step'] = 0
    ema = {k: sd[k].clone() for k in names}
    ema['num_updates'] = 0
    osde = S.SubVP(0.1, 20., 1000)
    data = torch.tensor(g['data'])
    idx = lambda n: torch.linspace(0, n - 1, min(48, n)).long()     # noqa: E731
    for s in range(STEPS):
        masks = torch.tensor(np.unpackbits(g[f's{s}_masks'], axis=-1)).reshape(5, B, 1024)
        loss, grads, total = T.train_step(sd, opt, ema, osde, data[s * B:(s + 1) * B], torch.tensor(g[f's{s}_t']),
                                          torch.tensor(g[f's{s}_z']), masks, int(g['step0']) + s)
        assert abs(float(loss) - float(g[f's{s}_loss'])) < 1e-5 * float(g[f's{s}_loss'])
        assert abs(float(total) - float(g[f's{s}_gnorm'])) < 1e-4 * float(g[f's{s}_gnorm'])
        for n, gr in grads.items():
            flat = gr.reshape(-1)
            assert float((flat[idx(flat.numel())] - torch.tensor(g[f's{s}_g_{n}'])).abs().max()) <= 1e-4 * float(flat.abs().max()) + 1e-9, n
    for n in names:
        d = (sd[n] - sd0[n]).reshape(-1)
        dmax = max(float(np.abs(g[f'dp_{n}']).max()), 1e-12)
        assert float((d[idx(d.numel())] - torch.tensor(g[f'dp_{n}'])).abs().max()) <= 2e-2 * dmax + 1e-12, n
        e = (ema[n] - sd0[n]).reshape(-1)
        assert float((e[idx(e.numel())] - torch.tensor(g[f'dema_{n}'])).abs().max()) <= 2e-2 * dmax + 1e-12, n


def test_training_oracle_auxiliary_loss_reproduces_reference():
    """oracle/train_ref.aux_loss against the REAL reference's step_fn(auxiliary_loss=True) (train_aux_golden.npz): the four
    loss values and sampled gradients (DDIM chain of three evaluations under autograd + LBS restatement)."""
    from dposer_b200 import synthetic
    from oracle import lbs_ref
    from oracle import score_ref as S
    from oracle import train_ref as T
    g = golden('train_aux_golden.npz')
    B, N = g['data'].shape[0], int(g['nsteps'])
    stats = np.load(os.path.join(os.path.dirname(synthetic.__file__), 'data', 'amass_stats.npz'))
    mean, std = torch.tensor(stats['mean_poses']), torch.tensor(stats['std_poses'])
    m = synthetic.make_body_tensors('smplx')

    def body_fn(pose):
        full = torch.cat([torch.zeros(B, 3), pose, torch.zeros(B, 99)], 1)
        return lbs_ref.body_forward(m, torch.zeros(B, m['shapedirs'].shape[2]), full)
    sd = S.make_state_dict(42)
    names = T.param_names(sd)
    leaves = {k: sd[k].clone().requires_grad_(True) for k in names}
    full = dict(sd)
    full.update(leaves)
    masks = torch.tensor(np.unpackbits(g['masks'], axis=-1)).reshape(N, 5, B, 1024)
    ol, osc, ov, oj = T.aux_loss(full, S.SubVP(0.1, 20., 1000), torch.tensor(g['data']), torch.tensor(g['t']), torch.tensor(g['z']),
                                 masks, 0.1, lambda v: v * std + mean, body_fn, N, reduce_mean=True)
    for a, k in ((ol, 'step_loss'), (osc, 'score_loss'), (ov, 'v2v_loss'), (oj, 'j2j_loss')):
        assert abs(float(a.detach()) - float(g[k])) <= 2e-5 * abs(float(g[k])), k
    used = [k for k in names if not k.startswith('pre_dense_cond')]
    og = dict(zip(used, torch.autograd.grad(ol, [leaves[k] for k in used])))
    idx = lambda n: torch.linspace(0, n - 1, min(48, n)).long()     # noqa: E731
    for n in used:
        flat = og[n].reshape(-1)
        assert float((flat[idx(flat.numel())] - torch.tensor(g[f'g_{n}'])).abs().max()) <= 2e-4 * float(g[f'gmax_{n}']) + 1e-10, n
