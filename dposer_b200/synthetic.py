"""Synthetic stand-ins for the assets that cannot ship (SURVEY.md 8d): random-init score
weights, SMPL / SMPL-X shaped body tensors, and the benchmark inputs derived from the AMASS
poses the reference does ship (examples/toy_data.npz, extracted to dposer_b200/data/).
Used by tests, bench.py and smoke() on both the GPU and the CPU-oracle side.
"""
import os
import types

import numpy as np
import torch

from .body_model import SMPL_PARENTS, SMPLX_PARENTS, SMPL_EXTRA_VIDS, SMPLX_EXTRA_VIDS

_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'data')


def default_config():
    """configs/subvp/amass_scorefc_continuous.py + configs/default_amass_configs.py values that the
    hot path reads (attribute-style object; ml_collections is not needed)."""
    ns = types.SimpleNamespace
    return ns(
        data=ns(normalize=True, rot_rep='axis', min_max=False),
        training=ns(sde='subvpsde', continuous=True, batch_size=1280, n_iters=400001, auxiliary_loss=False, denoise_steps=10,
                    likelihood_weighting=False, reduce_mean=True),
        optim=ns(weight_decay=0, optimizer='Adam', lr=2e-4, beta1=0.9, eps=1e-8, warmup=5000, grad_clip=1.),
        sampling=ns(method='pc', predictor='euler_maruyama', corrector='none', n_steps_each=1, noise_removal=True,
                    probability_flow=False, snr=0.16),
        model=ns(type='ScoreModelFC', HIDDEN_DIM=1024, EMBED_DIM=512, N_BLOCKS=2, dropout=0.1, fourier_scale=16,
                 scale_by_sigma=True, ema_rate=0.9999, nonlinearity='swish', embedding_type='positional',
                 sigma_min=0.01, sigma_max=50, num_scales=1000, beta_min=0.1, beta_max=20.),
        eval=ns(batch_size=50, num_samples=500),
        seed=42,
        device=torch.device('cuda:0') if torch.cuda.is_available() else torch.device('cpu'),
    )


def make_score_model(seed=42, config=None, pose_dim=3):
    """SURVEY 8(d) "Score weights": default init under torch.manual_seed(seed) in the reference's module
    order, then every GroupNorm weight~U(0.5,1.5), bias~N(0,0.1^2) (same generator, module order).
    pose_dim=3: the 63-D axis-angle network; pose_dim=6: the 126-D rot6d one."""
    from .model import ScoreModelFC
    config = config or default_config()
    torch.manual_seed(seed)
    m = ScoreModelFC(config, n_poses=21, pose_dim=pose_dim, hidden_dim=1024, embed_dim=512, n_blocks=2)
    for mod in m.modules():
        if isinstance(mod, torch.nn.GroupNorm):
            with torch.no_grad():
                mod.weight.copy_(torch.rand(1024) + 0.5)
                mod.bias.copy_(torch.randn(1024) * 0.1)
    return m.eval()


def toy_poses():
    return torch.tensor(np.load(os.path.join(_DATA, 'toy_poses.npz'))['pose_samples'])      # [500,63] AMASS


def gesture_sequences():
    d = np.load(os.path.join(_DATA, 'gestures.npz'))
    return torch.tensor(d['pose_body']), torch.tensor(d['root_orient'])                     # [240,63], [240,3]


def make_body_tensors(model_type='smpl', seed=None, nnz=4, reg_nnz=32):
    """Random body model with SMPL (6890/24/10) or SMPL-X (10475/55/20) shapes -- recipe of SURVEY 8(d) c2/c4."""
    if model_type == 'smpl':
        V, J, S, parents, extra = 6890, 24, 10, SMPL_PARENTS, SMPL_EXTRA_VIDS
        seed = 7 if seed is None else seed
    elif model_type == 'smplx':
        V, J, S, parents, extra = 10475, 55, 20, SMPLX_PARENTS, SMPLX_EXTRA_VIDS
        seed = 8 if seed is None else seed
    else:
        raise ValueError(model_type)
    g = torch.Generator().manual_seed(seed)
    lo = torch.tensor([-0.9, -1.2, -0.2])
    hi = torch.tensor([0.9, 0.6, 0.2])
    v_template = lo + (hi - lo) * torch.rand(V, 3, generator=g)
    shapedirs = torch.randn(V, 3, S, generator=g) * 0.01
    posedirs = torch.randn((J - 1) * 9, V * 3, generator=g) * 2e-3

    def dirichlet(rows, k):
        e = -torch.log(torch.rand(rows, k, generator=g).clamp_min(1e-12))
        return e / e.sum(1, keepdim=True)
    J_regressor = torch.zeros(J, V)
    for j in range(J):
        idx = torch.randperm(V, generator=g)[:reg_nnz]
        J_regressor[j, idx] = dirichlet(1, reg_nnz)[0]
    lbs_weights = torch.zeros(V, J)
    cols = torch.stack([torch.randperm(J, generator=g)[:nnz] for _ in range(V)])
    lbs_weights.scatter_(1, cols, dirichlet(V, nnz))
    out = dict(v_template=v_template, shapedirs=shapedirs, posedirs=posedirs, J_regressor=J_regressor,
               lbs_weights=lbs_weights, parents=list(parents), extra_vids=list(extra),
               faces=torch.randint(0, V, (2 * V, 3), generator=g))
    if model_type == 'smplx':
        out['lmk_faces'] = torch.randint(0, V, (51, 3), generator=g).to(torch.int32)
        out['lmk_bary'] = dirichlet(51, 3)
        # smplx model files carry hands_meanl / hands_meanr (45 each); lib/body_model/smpl.py's SMPLX runs with the
        # smplx defaults (flat_hand_mean=False) so this constant NON-ZERO hand pose is part of every forward.
        # Separate generator: the tensors above stay bit-identical to the round-1 recipe.
        out['hands_mean'] = 0.2 * torch.randn(90, generator=torch.Generator().manual_seed(seed + 1000))
    return out


def lbs_inputs(B, model_type='smpl', seed=11):
    """c2 inputs: AMASS toy poses tiled to B + N(0,0.05^2) jitter (hands zero), root/betas/trans ~ N(0,1)."""
    g = torch.Generator().manual_seed(seed)
    toy = toy_poses()
    reps = (B + toy.shape[0] - 1) // toy.shape[0]
    body = toy.repeat(reps, 1)[:B] + 0.05 * torch.randn(B, 63, generator=g)
    root = torch.randn(B, 3, generator=g)
    trans = torch.randn(B, 3, generator=g)
    if model_type == 'smpl':
        betas = torch.randn(B, 10, generator=g)
        pose_body = torch.cat([body, torch.zeros(B, 6)], dim=1)           # [B,69], hand joints zero
        return dict(root_orient=root, pose_body=pose_body, betas=betas, trans=trans)
    betas = torch.randn(B, 10, generator=g)
    return dict(root_orient=root, pose_body=body, betas=betas, trans=trans)


def full_pose_from(inputs, model_type='smpl'):
    """The concatenated [B, J*3] pose / [B,S] shape the oracle's body_forward takes."""
    B = inputs['pose_body'].shape[0]
    if model_type == 'smpl':
        return torch.cat([inputs['root_orient'], inputs['pose_body']], dim=1), inputs['betas']
    pose = torch.cat([inputs['root_orient'], inputs['pose_body'], torch.zeros(B, 9 + 90)], dim=1)
    return pose, torch.cat([inputs['betas'], torch.zeros(B, 10)], dim=1)


def uv_sphere(n_rings=82, n_lon=84, radius=1.0, center=(0., 0., 0.)):
    """Closed UV sphere: two poles and n_rings rings of n_lon vertices, faces wound outward.  The defaults give
    SMPL's counts (V = 6890, F = 13776); (101, 104) gives V = 10506, F = 21008 (more faces than SMPL-X's 20908).
    Returns fp32 vertices [V,3] and int32 faces [2 n_lon n_rings, 3] as numpy arrays."""
    th = np.pi * np.arange(1, n_rings + 1) / (n_rings + 1)
    ph = 2 * np.pi * np.arange(n_lon) / n_lon
    ring = np.stack([np.sin(th)[:, None] * np.cos(ph), np.sin(th)[:, None] * np.sin(ph),
                     np.repeat(np.cos(th)[:, None], n_lon, 1)], -1).reshape(-1, 3)
    v = np.concatenate([[[0., 0., 1.]], ring, [[0., 0., -1.]]]) * radius + np.asarray(center)
    r = lambda i, j: 1 + i * n_lon + (j % n_lon)                           # noqa: E731  ring i (0-based), longitude j
    j = np.arange(n_lon)
    south = 1 + n_rings * n_lon
    faces = [np.stack([np.zeros(n_lon, int), r(0, j), r(0, j + 1)], 1)]
    for i in range(n_rings - 1):
        a, b, c, d = r(i, j), r(i + 1, j), r(i + 1, j + 1), r(i, j + 1)
        faces += [np.stack([a, b, c], 1), np.stack([a, c, d], 1)]
    faces.append(np.stack([np.full(n_lon, south), r(n_rings - 1, j + 1), r(n_rings - 1, j)], 1))
    return v.astype(np.float32), np.concatenate(faces).astype(np.int32)


def dented_sphere(depth, seed, n_rings=82, n_lon=84, cap_deg=(65., 80.), jitter=0.01):
    """A UV sphere with a seeded cap pushed inward: cap height h (along a random axis u) becomes h (1 - 2 depth w),
    w = 1 inside cap_deg[0] and a smoothstep to 0 at cap_deg[1].  depth = 0: the sphere; depth = 0.5 flattens the
    cap onto the equatorial plane; depth = 1 mirrors it onto the opposite wall, where the two sheets interpenetrate
    wherever the jitter crosses (the most self-intersection); depth > 1 pushes it through the wall.  Before the dent
    every vertex moves radially by a smooth seeded field of amplitude `jitter` (a few low-frequency waves), so that
    no pair of faces is exactly degenerate.  Returns fp32 vertices [V,3] (the faces are uv_sphere's)."""
    v, _ = uv_sphere(n_rings, n_lon)
    g = np.random.default_rng(seed)
    p = v.astype(np.float64)
    rad = np.zeros(len(p))
    for _ in range(4):
        k = g.normal(size=3)
        k *= g.uniform(10., 24.) / np.linalg.norm(k)
        rad += g.uniform(0.5, 1.) * np.sin(p @ k + g.uniform(0, 2 * np.pi))
    p *= (1 + jitter * rad / 4)[:, None]
    u = g.normal(size=3)
    u /= np.linalg.norm(u)
    h = p @ u
    c_in, c_out = np.cos(np.radians(cap_deg[0])), np.cos(np.radians(cap_deg[1]))
    t = np.clip((h / np.linalg.norm(p, axis=1) - c_out) / (c_in - c_out), 0, 1)
    w = t * t * (3 - 2 * t)
    p -= (2 * depth * w * h)[:, None] * u
    return p.astype(np.float32)


def two_spheres(n_rings=40, n_lon=48, offset=1.0):
    """Two overlapping unit UV spheres (centres `offset` apart along x) as one two-component mesh."""
    v0, f0 = uv_sphere(n_rings, n_lon, center=(0., 0., 0.))
    v1, f1 = uv_sphere(n_rings, n_lon, center=(offset, 0.01, 0.02))
    return np.concatenate([v0, v1]), np.concatenate([f0, f1 + len(v0)]).astype(np.int32)


def completion_inputs(n_partial=4096, hypotheses=10, seed=21, normalizer=None):
    """c3 inputs: normalised toy poses tiled (+N(0,0.05^2)), legs masked, x hypotheses."""
    from .misc import create_mask, Posenormalizer
    normalizer = normalizer or Posenormalizer(None, device='cpu', normalize=True, min_max=False, rot_rep='axis')
    g = torch.Generator().manual_seed(seed)
    toy = normalizer.offline_normalize(toy_poses())
    reps = (n_partial + toy.shape[0] - 1) // toy.shape[0]
    poses = toy.repeat(reps, 1)[:n_partial] + 0.05 * torch.randn(n_partial, 63, generator=g)
    torch.manual_seed(seed)
    mask, obs = create_mask(poses, part='legs')
    return poses, mask.repeat(hypotheses, 1), obs.repeat(hypotheses, 1)
