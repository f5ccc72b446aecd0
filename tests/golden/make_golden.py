#!/usr/bin/env python
"""Generate golden fixtures by running the REAL reference (imported from /root/reference).

Run in the build container only (the GPU box has no /root/reference):
    python tests/golden/make_golden.py
Writes small .npz files next to this script plus the shipped-data extracts under
dposer_b200/data/.  While generating, it also asserts that oracle/ reproduces the
reference (so a fixture is only ever written from a state where oracle == reference).
Import shims follow SURVEY.md Appendix C (test-only scaffolding around the untouched reference).
"""
import math
import os
import sys
import types
from unittest.mock import MagicMock

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = '/root/reference'
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)

for n in ['torchgeometry', 'smplx', 'smplx.utils', 'smplx.body_models', 'pyrender', 'trimesh', 'matplotlib',
          'matplotlib.pyplot', 'pymeshlab', 'plyfile', 'tensorboardX', 'pytorch3d', 'pytorch3d.renderer',
          'pytorch3d.structures']:
    sys.modules[n] = MagicMock()
mc = types.ModuleType('ml_collections')


class ConfigDict(dict):
    __getattr__ = dict.__getitem__
    __setattr__ = dict.__setitem__


mc.ConfigDict = ConfigDict
sys.modules['ml_collections'] = mc
from absl import flags  # noqa: E402

cf = types.ModuleType('ml_collections.config_flags')
cf.config_flags = types.SimpleNamespace(
    DEFINE_config_file=lambda name, default, help, lock_config=False:
    (name in flags.FLAGS) or flags.DEFINE_string(name, default, help))
sys.modules['ml_collections.config_flags'] = cf

from configs.subvp.amass_scorefc_continuous import get_config  # noqa: E402
from lib.algorithms.advanced import sde_lib, sampling  # noqa: E402
from lib.algorithms.advanced import utils as mutils  # noqa: E402
from lib.algorithms.advanced.model import ScoreModelFC, get_timestep_embedding  # noqa: E402
from lib.body_model import constants, fitting_losses  # noqa: E402
from lib.body_model.utils import BodyPartIndices, BodySegIndices  # noqa: E402
from lib.dataset.AMASS import Posenormalizer  # noqa: E402
from lib.dataset.EvaSampler import DistributedEvalSampler  # noqa: E402
from lib.utils.misc import create_mask, gaussian_smoothing  # noqa: E402
from run.completion import DPoserComp  # noqa: E402
from run.motion_denoising import MotionDenoise  # noqa: E402

from oracle import score_ref as S  # noqa: E402
from oracle import fitting_ref as Fr  # noqa: E402

torch.set_grad_enabled(True)


def close(a, b, tol, what):
    a, b = torch.as_tensor(a), torch.as_tensor(b)
    err = (a - b).abs().max().item()
    scale = max(b.abs().max().item(), 1e-30)
    assert err <= tol * scale, f'{what}: oracle != reference, err {err:.3e} scale {scale:.3e}'
    print(f'  ok {what}: max err {err:.2e} (scale {scale:.2e})')


def build_reference_model(cfg):
    """SURVEY 8(d) "Score weights" recipe on the REAL reference class."""
    torch.manual_seed(42)
    m = ScoreModelFC(cfg, n_poses=21, pose_dim=3, hidden_dim=1024, embed_dim=512, n_blocks=2)
    for mod in m.modules():
        if isinstance(mod, torch.nn.GroupNorm):
            with torch.no_grad():
                mod.weight.copy_(torch.rand(1024) + 0.5)
                mod.bias.copy_(torch.randn(1024) * 0.1)
    return m.eval()


def main():
    cfg = get_config()
    cfg.device = torch.device('cpu')
    model = build_reference_model(cfg)
    ref_sd = {k: v.detach() for k, v in model.state_dict().items()}
    sd = S.make_state_dict(42)
    # --- weights: same recipe must give the same tensors (bit-exact)
    fingerprint = {}
    for k, v in ref_sd.items():
        if k.startswith('pre_dense_cond'):
            continue
        assert torch.equal(v, sd[k]), f'weight recipe mismatch at {k}'
        # exactly rounded sum: torch's CPU sum() splits the reduction by thread count, so it can differ in the last
        # bit from one host to another
        fingerprint[k] = np.float64(math.fsum(v.double().abs().flatten().tolist()))
    print('weights: oracle recipe == reference recipe (bit-exact), params',
          sum(v.numel() for k, v in ref_sd.items() if k != 'sigmas'))
    np.savez(os.path.join(HERE, 'weights_fingerprint.npz'), **fingerprint)

    sde = sde_lib.subVPSDE(beta_min=0.1, beta_max=20., N=1000)
    osde = S.SubVP(0.1, 20., 1000)
    score_fn = mutils.get_score_fn(sde, model, train=False, continuous=True)

    # --- known-answer scalars (SURVEY Appendix D)
    ts = torch.linspace(1, 1e-3, 1000)
    idx = torch.tensor([0, 499, 500, 998, 999])
    t5 = ts[idx]
    _, g = sde.sde(torch.zeros(5, 1), t5)
    alpha, std = sde.return_alpha_sigma(t5)
    labels = t5 * 999
    kat = dict(i=idx.numpy(), t=t5.numpy(), label=labels.numpy(), idx=labels.long().numpy(), g=g.numpy(),
               alpha=alpha[:, 0].numpy(), std=std.numpy(), sigmas=model.sigmas[labels.long()].numpy(),
               temb_4995=get_timestep_embedding(torch.tensor([499.5]), 512)[0].numpy(),
               sde_alphas=sde.alphas.numpy(), all_idx=(ts * 999).long().numpy())
    close(osde.sde(torch.zeros(5, 1), t5)[1], g, 0, 'g(t)')
    close(osde.alpha_sigma(t5)[1], std, 0, 'std(t)')
    close(S.timestep_embedding(torch.tensor([499.5])), kat['temb_4995'][None], 0, 'temb')
    close(S.sigma_table(), model.sigmas, 0, 'sigmas')
    np.savez(os.path.join(HERE, 'known_answers.npz'), **kat)

    # --- score net / score fn
    toy = np.load(os.path.join(REF, 'examples/toy_data.npz'))['pose_samples']
    stats = torch.load(os.path.join(REF, 'data/AMASS/amass_processed/version1/train/axis_normalize2.pt'))
    stats1 = torch.load(os.path.join(REF, 'data/AMASS/amass_processed/version1/train/axis_normalize1.pt'))
    os.makedirs(os.path.join(ROOT, 'dposer_b200/data'), exist_ok=True)
    np.savez(os.path.join(ROOT, 'dposer_b200/data/amass_stats.npz'),
             mean_poses=stats['mean_poses'].numpy(), std_poses=stats['std_poses'].numpy(),
             min_poses=stats1['min_poses'].numpy(), max_poses=stats1['max_poses'].numpy())
    np.savez_compressed(os.path.join(ROOT, 'dposer_b200/data/toy_poses.npz'), pose_samples=toy)
    ges = np.load(os.path.join(REF, 'examples/Gestures_3_poses_batch005.npz'))
    np.savez_compressed(os.path.join(ROOT, 'dposer_b200/data/gestures.npz'),
                        pose_body=ges['pose_body'].astype(np.float32),
                        root_orient=ges['root_orient'].astype(np.float32))
    mean_params = np.load(os.path.join(REF, 'lib/body_model/smpl_mean_params.npz'))
    np.savez(os.path.join(ROOT, 'dposer_b200/data/smpl_mean_params.npz'), **{k: mean_params[k] for k in mean_params.files})

    norm = Posenormalizer(os.path.join(REF, 'data/AMASS/amass_processed/version1/train'), device='cpu',
                          normalize=True, min_max=False, rot_rep='axis')
    g_ = torch.Generator().manual_seed(5)
    x7 = norm.offline_normalize(torch.tensor(toy[:7])) + 0.3 * torch.randn(7, 63, generator=g_)
    close(Fr.normalize(torch.tensor(toy[:7]), stats['mean_poses'], stats['std_poses']),
          norm.offline_normalize(torch.tensor(toy[:7])), 0, 'normalize')
    close(Fr.denormalize(x7, stats['mean_poses'], stats['std_poses']), norm.offline_denormalize(x7), 0, 'denormalize')
    score_out, model_out = {}, {}
    with torch.no_grad():
        for tv in [1.0, 0.5, 0.1, 0.01, 1e-3]:
            vt = torch.ones(7) * tv
            score_out[f'{tv}'] = score_fn(x7, vt, None, None).numpy()
            model_out[f'{tv}'] = model(x7, vt * 999).numpy()
            close(S.score_fn(sd, osde, x7, vt), score_out[f'{tv}'], 2e-6, f'score_fn t={tv}')
            close(S.score_model_forward(sd, x7, vt * 999), model_out[f'{tv}'], 2e-6, f'model t={tv}')
        # per-row t (general forward)
        vt = torch.tensor([1.0, 0.73, 0.5, 0.31, 0.1, 0.01, 1e-3])
        model_out['mixed'] = model(x7, vt * 999).numpy()
        score_out['mixed'] = score_fn(x7, vt, None, None).numpy()
        close(S.score_model_forward(sd, x7, vt * 999), model_out['mixed'], 2e-6, 'model mixed t')
    np.savez(os.path.join(HERE, 'score_golden.npz'), x=x7.numpy(), t_mixed=vt.numpy(),
             **{f'score_{k}': v for k, v in score_out.items()}, **{f'model_{k}': v for k, v in model_out.items()})

    # --- samplers (reference draws from torch's global CPU generator; we replay the draws)
    samp = {}
    for name, N, corr, task, pf, start in [('em8', 8, 'none', None, False, 0), ('em32', 32, 'none', None, False, 0),
                                           ('lang8', 1000, 'langevin', 'denoise', False, 992),
                                           ('comp8', 8, 'none', 'completion', False, 0),
                                           ('ode8', 8, 'none', None, True, 0),
                                           ('den16', 16, 'none', 'denoise', False, 10)]:
        B = 5
        cfg.sampling.corrector = corr
        cfg.sampling.probability_flow = pf
        rsde = sde_lib.subVPSDE(0.1, 20., N=N)
        fn = sampling.get_sampling_fn(cfg, rsde, (B, 63), lambda x: x, 1e-3, device='cpu')
        gz = torch.Generator().manual_seed(77)
        z0 = torch.randn(B, 63, generator=gz)
        obs = mask = None
        args = None
        if task == 'completion':
            torch.manual_seed(3)
            mask, obs = create_mask(norm.offline_normalize(torch.tensor(toy[:B])), part='legs')
            args = types.SimpleNamespace(task='completion')
        if task == 'denoise':
            args = types.SimpleNamespace(task='denoise')
        torch.manual_seed(1234)
        traj, out = fn(model, observation=obs, mask=mask, z=z0.clone(), start_step=start, args=args)
        # replay the draws in the reference's order (sampling.py:459-460, 282-302, 413-422, 182-188)
        torch.manual_seed(1234)
        noise = []
        for i in range(start, N):
            d = {}
            if corr == 'langevin':
                d['corr'] = torch.randn(B, 63)
            if task == 'completion':
                d['imp_c'] = torch.randn(B, 63)
            d['pred'] = torch.randn(B, 63)
            if task == 'completion':
                d['imp_p'] = torch.randn(B, 63)
            noise.append(d)
        noise_by_step = {start + i: d for i, d in enumerate(noise)}
        otraj, oout = S.pc_sample(sd, S.SubVP(0.1, 20., N), z0, 1e-3, noise=noise_by_step, corrector=corr,
                                  observation=obs, mask=mask, task=task, start_step=start,
                                  probability_flow=pf, keep_traj=True)
        close(oout, out, 2e-5, f'pc_sampler {name} x_mean')
        close(otraj, traj, 2e-5, f'pc_sampler {name} traj')
        samp[f'{name}_z0'] = z0.numpy()
        samp[f'{name}_out'] = out.numpy()
        samp[f'{name}_traj_last'] = traj[-1].numpy()
        for k in ['pred', 'corr', 'imp_c', 'imp_p']:
            if k in noise[0]:
                samp[f'{name}_noise_{k}'] = torch.stack([d[k] for d in noise]).numpy()
        if obs is not None:
            samp[f'{name}_obs'] = obs.numpy()
            samp[f'{name}_mask'] = mask.numpy()
    cfg.sampling.corrector = 'none'
    cfg.sampling.probability_flow = False
    np.savez(os.path.join(HERE, 'sampler_golden.npz'), **samp)

    # --- prior loss (completion: mean, weighted by accident; denoise: sum/B unweighted; smplify: sum/B weighted)
    pl = {}
    comp = DPoserComp(model, sde, True, batch_size=7)
    timesteps = torch.linspace(1, 1e-3, 1000)
    for name, qt in [('q799', 799), ('q998', 998), ('q400', 400)]:
        x0 = x7.clone().requires_grad_(True)
        vt = torch.ones(7) * timesteps[qt]
        torch.manual_seed(9)
        loss = comp.loss(x0, vt, qt)                 # 3rd positional -> weighted (SURVEY B-3)
        loss.backward()
        torch.manual_seed(9)
        z = torch.randn(7, 63)
        ol, og = S.prior_loss(sd, osde, x7, vt, z, weighted=True, reduce='mean')
        close(ol, loss.detach(), 2e-5, f'prior loss {name}')
        close(og, x0.grad, 2e-5, f'prior grad {name}')
        pl[f'{name}_z'] = z.numpy()
        pl[f'{name}_loss'] = loss.detach().numpy()
        pl[f'{name}_grad'] = x0.grad.numpy()
    # motion-denoise flavour via the real class method (unbound: only needs sde/rsde/loss_fn/batch_size)
    md = types.SimpleNamespace(sde=sde, rsde=comp.rsde, loss_fn=comp.loss_fn, batch_size=7, score_fn=comp.score_fn)
    md.one_step_denoise = types.MethodType(MotionDenoise.one_step_denoise, md)
    md.multi_step_denoise = types.MethodType(MotionDenoise.multi_step_denoise, md)
    for name, weighted, multi in [('md_plain', False, False), ('md_weighted', True, False), ('md_ddim', False, True)]:
        x0 = x7.clone().requires_grad_(True)
        vt = torch.ones(7) * timesteps[450]
        torch.manual_seed(10)
        loss = MotionDenoise.DPoser_loss(md, x0, vt, 450, weighted=weighted, multi_denoise=multi)
        loss.backward()
        torch.manual_seed(10)
        z = torch.randn(7, 63)
        ol, og = S.prior_loss(sd, osde, x7, vt, z, weighted=weighted, reduce='sum', divisor=7, multi_denoise=multi)
        close(ol, loss.detach(), 2e-5, f'prior loss {name}')
        close(og, x0.grad, 2e-5, f'prior grad {name}')
        pl[f'{name}_z'] = z.numpy()
        pl[f'{name}_loss'] = loss.detach().numpy()
        pl[f'{name}_grad'] = x0.grad.numpy()
    pl['x0'] = x7.numpy()
    np.savez(os.path.join(HERE, 'prior_golden.npz'), **pl)

    # --- integer tables
    ints = {}
    for part in ['legs', 'arms', 'trunk', 'hands', 'left_leg', 'right_leg', 'left_arm', 'right_arm']:
        ints[f'part_{part}'] = np.array(getattr(BodyPartIndices, part))
        ints[f'seg_{part}'] = np.array(getattr(BodySegIndices, part))
        m, _ = create_mask(torch.zeros(2, 63), part=part)
        ints[f'maskzero_{part}'] = np.nonzero(m[0].numpy() == 0)[0]
        assert np.array_equal(ints[f'maskzero_{part}'], np.sort(Fr.mask_indices(part).numpy()))
        assert Fr.BODY_PARTS[part] == list(getattr(BodyPartIndices, part))
    joints = [constants.JOINT_MAP[i] for i in constants.JOINT_NAMES]
    joints[:25] = [55, 12, 17, 19, 21, 16, 18, 20, 0, 2, 5, 8, 1, 4, 7, 56, 57, 58, 59, 60, 61, 62, 63, 64, 65]
    ints['smplx_joint_map49'] = np.array(joints)          # lib/body_model/smpl.py:53-58
    ints['op_ind'] = np.array([constants.JOINT_IDS[j] for j in ['OP RHip', 'OP LHip', 'OP RShoulder', 'OP LShoulder']])
    ints['gt_ind'] = np.array([constants.JOINT_IDS[j] for j in ['Right Hip', 'Left Hip', 'Right Shoulder', 'Left Shoulder']])
    for N, total, trun, off, nm in [(1000, 200, 5.0, 2, 'completion'), (500, 180, 4.0, 2, 'denoise'), (500, 500, 20.0, 5, 'smplify')]:
        ints[f'quan_t_{nm}'] = np.array(S.quan_t_schedule(N, total, trun, off))
    shard = []
    for total, world in [(500, 1), (500, 8), (4096, 8), (13, 4), (5, 8), (40960, 3), (8192, 7)]:
        for r in range(world):
            smp = DistributedEvalSampler(list(range(total)), num_replicas=world, rank=r)
            ix = list(iter(smp))
            st, n = Fr.shard_range(total, world, r)
            assert ix == list(range(st, st + n)), (total, world, r)
            shard.append([total, world, r, ix[0] if ix else -1, len(ix)])
    ints['shards'] = np.array(shard)
    np.savez(os.path.join(HERE, 'int_tables.npz'), **ints)
    print('int tables ok; quan_t completion', ints['quan_t_completion'][[0, -1]], 'denoise',
          ints['quan_t_denoise'][[0, -1]], 'smplify', ints['quan_t_smplify'][[0, -1]])

    # --- fitting losses, smoothing
    gen = torch.Generator().manual_seed(123)
    B = 6
    jts = torch.randn(B, 49, 3, generator=gen) * 0.3 + torch.tensor([0., 0., 30.])
    kp = torch.randn(B, 49, 2, generator=gen) * 50 + 512
    conf = torch.rand(B, 49, generator=gen)
    conf[:, 25:] = 0
    conf[1, 9] = 0
    pose = torch.randn(B, 63, generator=gen) * 0.3
    betas = torch.randn(B, 10, generator=gen)
    cam_t = torch.randn(B, 3, generator=gen)
    cam_est = torch.randn(B, 3, generator=gen)
    center = torch.full((B, 2), 512.)
    prior = torch.tensor(3.7)
    ref_body = fitting_losses.body_fitting_loss(pose, betas, jts, cam_t, center, kp, conf,
                                                lambda p, b, q: prior, 480, focal_length=5000., verbose=False)
    ref_cam = fitting_losses.camera_fitting_loss(jts, cam_t, cam_est, center, kp, conf, focal_length=5000.)
    close(Fr.body_fitting_loss(pose, betas, jts, center, kp, conf, prior), ref_body, 1e-6, 'body_fitting_loss')
    close(Fr.camera_fitting_loss(jts, cam_t, cam_est, center, kp, conf, op_ind=ints['op_ind'], gt_ind=ints['gt_ind']),
          ref_cam, 1e-6, 'camera_fitting_loss')
    sm_in = torch.randn(60, 63, generator=gen)
    ref_sm = gaussian_smoothing(sm_in, 3, 2)
    close(Fr.gaussian_smoothing(sm_in, 3, 2), ref_sm, 1e-6, 'gaussian_smoothing')
    np.savez(os.path.join(HERE, 'fitting_golden.npz'), joints=jts.numpy(), kp=kp.numpy(), conf=conf.numpy(),
             pose=pose.numpy(), betas=betas.numpy(), cam_t=cam_t.numpy(), cam_est=cam_est.numpy(),
             body_loss=ref_body.numpy(), cam_loss=ref_cam.numpy(), prior=prior.numpy(),
             smooth_in=sm_in.numpy(), smooth_out=ref_sm.numpy())
    # APD is defined in lib/utils/metric.py which imports pymeshlab (mocked) -> import works
    from lib.utils.metric import average_pairwise_distance
    j3 = torch.randn(12, 22, 3, generator=gen)
    ref_apd = average_pairwise_distance(j3)
    close(Fr.apd(j3), ref_apd, 1e-6, 'APD')
    np.savez(os.path.join(HERE, 'apd_golden.npz'), joints=j3.numpy(), apd=ref_apd.numpy())
    print('all golden fixtures written to', HERE)


if __name__ == '__main__':
    main()
