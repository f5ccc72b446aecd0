"""Small host-side helpers of the hot path (reference lib/utils/misc.py, lib/body_model/utils.py,
lib/dataset/AMASS.py:187-259, lib/dataset/EvaSampler.py).  Pure tensor bookkeeping -- device agnostic."""
import math
import os

import numpy as np
import torch
import torch.nn.functional as F

N_POSES = 21
_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'data')

_BODY_JOINT_NAMES = ['pelvis', 'left_hip', 'right_hip', 'spine1', 'left_knee', 'right_knee', 'spine2', 'left_ankle',
                     'right_ankle', 'spine3', 'left_foot', 'right_foot', 'neck', 'left_collar', 'right_collar',
                     'head', 'left_shoulder', 'right_shoulder', 'left_elbow', 'right_elbow', 'left_wrist',
                     'right_wrist']
_IDX = {n: i - 1 for i, n in enumerate(_BODY_JOINT_NAMES)}      # pelvis excluded (lib/body_model/utils.py:36)


class BodyPartIndices:
    """lib/body_model/utils.py:39-47 (integer tables, bit-exact)."""
    left_leg = sorted(_IDX[n] for n in ['left_hip', 'left_knee', 'left_ankle', 'left_foot'])
    right_leg = sorted(_IDX[n] for n in ['right_hip', 'right_knee', 'right_ankle', 'right_foot'])
    left_arm = sorted(_IDX[n] for n in ['left_collar', 'left_shoulder', 'left_elbow', 'left_wrist'])
    right_arm = sorted(_IDX[n] for n in ['right_collar', 'right_shoulder', 'right_elbow', 'right_wrist'])
    trunk = sorted(_IDX[n] for n in ['spine1', 'spine2', 'spine3', 'left_shoulder', 'right_shoulder'])
    hands = sorted(_IDX[n] for n in ['left_wrist', 'right_wrist'])
    legs = sorted(left_leg + right_leg)
    arms = sorted(left_arm + right_arm)


def create_mask(body_poses, part='legs', observation_type='noise'):
    """lib/utils/misc.py:27-55: 0/1 mask (0 on the part's dims) and the observation with those dims noise-filled."""
    assert len(body_poses.shape) == 2 and body_poses.shape[1] % N_POSES == 0
    rot_n = body_poses.shape[1] // N_POSES
    assert rot_n in [3, 6]
    joints = getattr(BodyPartIndices, part)
    idx = (torch.tensor(joints).view(-1, 1) * rot_n + torch.arange(rot_n).view(1, -1)).flatten()
    mask = body_poses.new_ones(body_poses.shape)
    mask[:, idx] = 0
    observation = body_poses.clone()
    if observation_type == 'noise':
        observation[:, idx] = torch.randn_like(observation[:, idx])
    else:
        # the SMPL mean pose on the masked joints (misc.py:43-53): 'pose'[6:] of the reference's smpl_mean_params.npz
        # (23 joints x rot6d), shipped in dposer_b200/data
        from .transforms import rot6d_to_axis_angle
        mean6 = torch.tensor(np.load(os.path.join(_DATA, 'smpl_mean_params.npz'))['pose'][6:], dtype=torch.float32,
                             device=body_poses.device)
        fill = rot6d_to_axis_angle(mean6.reshape(-1, 6)).reshape(-1) if rot_n == 3 else mean6
        observation[:, idx] = fill[None, idx].repeat(body_poses.shape[0], 1)
    return mask, observation


def linear_interpolation(A, B, frames):
    """lib/utils/misc.py:58-61."""
    alpha = torch.linspace(0, 1, frames, device=A.device)[:, None]
    return (1 - alpha) * A + alpha * B


def gaussian_smoothing(data, window_size, sigma):
    """lib/utils/misc.py:84-95 (zero-padded conv1d along dim 0)."""
    k = torch.arange(window_size).float() - window_size // 2
    k = torch.exp(-0.5 * (k / sigma) ** 2)
    k = (k / k.sum()).view(1, 1, -1).to(data.device)
    d = data.transpose(0, 1).unsqueeze(1)
    return F.conv1d(d, k, padding=window_size // 2).squeeze(1).transpose(0, 1)


class Posenormalizer:
    """lib/dataset/AMASS.py:187-259.  ``data_path`` may be the reference's ``.../train`` directory (with
    {axis,rot6d}_normalize{1,2}.pt) or None for the AMASS statistics shipped in dposer_b200/data/amass_stats[_rot6d].npz
    (extracted from the reference's own files).  ``rot_rep='rot6d'`` normalises 126-D poses (``from_axis`` / ``to_axis``
    convert at the boundary, AMASS.py:200-201,254-256); the score-net kernels run 63-D (axis) and 126-D (rot6d) networks."""

    def __init__(self, data_path=None, device='cuda:0', normalize=True, min_max=True, rot_rep=None):
        assert rot_rep in ['rot6d', 'axis']
        self.normalize, self.min_max, self.rot_rep = normalize, min_max, rot_rep
        if data_path is not None and os.path.exists(os.path.join(data_path, f'{rot_rep}_normalize1.pt')):
            p1 = torch.load(os.path.join(data_path, f'{rot_rep}_normalize1.pt'))
            p2 = torch.load(os.path.join(data_path, f'{rot_rep}_normalize2.pt'))
            vals = [p1['min_poses'], p1['max_poses'], p2['mean_poses'], p2['std_poses']]
        else:
            s = np.load(os.path.join(_DATA, 'amass_stats.npz' if rot_rep == 'axis' else 'amass_stats_rot6d.npz'))
            vals = [torch.tensor(s[k]) for k in ('min_poses', 'max_poses', 'mean_poses', 'std_poses')]
        self.min_poses, self.max_poses, self.mean_poses, self.std_poses = [v.to(device) for v in vals]

    def _stats(self, poses, a, b):
        a, b = a.view(1, -1), b.view(1, -1)
        if len(poses.shape) == 3:
            a, b = a.unsqueeze(0), b.unsqueeze(0)
        return a, b

    def offline_normalize(self, poses, from_axis=False):
        assert len(poses.shape) in (2, 3)
        if from_axis and self.rot_rep == 'rot6d':
            from .transforms import axis_angle_to_rot6d
            poses = axis_angle_to_rot6d(poses.reshape(-1, 3)).reshape(*poses.shape[:-1], -1)
        if not self.normalize:
            return poses
        if self.min_max:
            lo, hi = self._stats(poses, self.min_poses, self.max_poses)
            return 2 * (poses - lo) / (hi - lo) - 1
        mean, std = self._stats(poses, self.mean_poses, self.std_poses)
        return (poses - mean) / std

    def column_affine(self):
        """(mean, std), one entry per column, with offline_normalize(poses) == (poses - mean) / std under the active
        rule: z-score as stored; min-max as mean = (lo + hi) / 2, std = (hi - lo) / 2; normalize=False as 0 / 1.
        The native fitting chains take this form (``steps.axis_to_rot6d_cols``)."""
        if not self.normalize:
            return torch.zeros_like(self.mean_poses), torch.ones_like(self.std_poses)
        if self.min_max:
            return (self.min_poses + self.max_poses) / 2, (self.max_poses - self.min_poses) / 2
        return self.mean_poses, self.std_poses

    def offline_denormalize(self, poses, to_axis=False):
        assert len(poses.shape) in (2, 3)
        if self.normalize:
            if self.min_max:
                lo, hi = self._stats(poses, self.min_poses, self.max_poses)
                poses = 0.5 * ((poses + 1) * (hi - lo) + 2 * lo)
            else:
                mean, std = self._stats(poses, self.mean_poses, self.std_poses)
                poses = poses * std + mean
        if to_axis and self.rot_rep == 'rot6d':
            from .transforms import rot6d_to_axis_angle
            poses = rot6d_to_axis_angle(poses.reshape(-1, 6)).reshape(*poses.shape[:-1], -1)
        return poses


def shard_range(total, num_replicas, rank):
    """Contiguous shard of ``DistributedEvalSampler`` (lib/dataset/EvaSampler.py:77-106):
    the first ``total % num_replicas`` ranks get one extra row.  Returns (start, count)."""
    base, mod = divmod(total, num_replicas)
    if rank <= mod:
        start = rank * (base + 1)
    else:
        start = mod * (base + 1) + (rank - mod) * base
    return start, (base + 1 if rank < mod else base)


def quan_t(strategy, N, total, step, trun, sample_time, offset):
    """Discrete time index of step ``step`` of ``total`` under a task loop's time strategy (run/completion.py:183-191,
    run/motion_denoising.py:240-247, run/smplify.py:153-166): '1' a uniform draw, '2' ``sample_time``, '3' the
    truncated linear schedule."""
    if strategy == '1':
        return int(torch.randint(N, [1]))
    if strategy == '2':
        return int(sample_time)
    if strategy == '3':
        return N - math.floor(torch.tensor(total - step - 1) * (N / (trun * total))) - offset
    raise NotImplementedError('unsupported time sampling strategy')


def quan_t_schedule(N, total_steps, trun, offset):
    """Every step's time index under strategy '3' (``quan_t``)."""
    return [quan_t('3', N, total_steps, s, trun, None, offset) for s in range(total_steps)]
