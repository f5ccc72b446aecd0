"""Rotation-representation helpers with the reference's names (lib/utils/transforms.py:197-255).

Data-preparation utilities (not on the hot path): plain torch ops on whatever device the input lives on.  The
reference builds them on third-party ``torchgeometry`` (``angle_axis_to_rotation_matrix`` /
``rotation_matrix_to_angle_axis``), which is not installable offline -- PARITY UNPINNED for those two legs: they are checked by
properties (round trips, orthonormality, agreement with the LBS oracle's Rodrigues) and against a restatement of
torchgeometry's published algorithms (oracle/tgm_ref.py); the Gram-Schmidt leg is pinned bit-exactly to the reference.
``misc.Posenormalizer(rot_rep='rot6d')`` and ``misc.create_mask(observation_type='mean')`` call them at the data boundary;
the score-net kernels take both representations (63-D axis, 126-D rot6d score networks: ``ScoreModelFC(config, 21, 6)``).
With a rot6d prior the native SMPLify / motion-denoising chains (``fitting.py``) do not call this module: the
axis -> rot6d map of ``axis_angle_to_rot6d`` and its Jacobian run as kernels inside the step
(``steps.axis_to_rot6d_cols`` / ``axis_to_rot6d_cols_vjp``), tested against float64 autograd through this function."""
import torch
import torch.nn.functional as F


def axis_angle_to_mat3x3(angle_axis):
    """[N,3] -> [N,3,3] (Rodrigues; first-order branch below 1e-6 rad like torchgeometry's Taylor branch)."""
    aa = angle_axis.reshape(-1, 3)
    theta = aa.norm(dim=1, keepdim=True)
    small = theta < 1e-6
    k = aa / theta.clamp_min(1e-12)
    kx, ky, kz = k[:, 0], k[:, 1], k[:, 2]
    z = torch.zeros_like(kx)
    K = torch.stack([z, -kz, ky, kz, z, -kx, -ky, kx, z], dim=1).reshape(-1, 3, 3)
    s, c = torch.sin(theta)[:, :, None], torch.cos(theta)[:, :, None]
    eye = torch.eye(3, dtype=aa.dtype, device=aa.device)[None]
    R = eye + s * K + (1 - c) * (K @ K)
    rx, ry, rz = aa[:, 0], aa[:, 1], aa[:, 2]
    one = torch.ones_like(rx)
    R1 = torch.stack([one, -rz, ry, rz, one, -rx, -ry, rx, one], dim=1).reshape(-1, 3, 3)
    return torch.where(small[:, :, None], R1, R)


def axis_angle_to_rot6d(angle_axis):
    """[N,3] -> [N,6]: the first two columns of the rotation matrix, row-major (transforms.py:237-252)."""
    return axis_angle_to_mat3x3(angle_axis)[:, :3, :2].reshape(-1, 6)


def rot6d_to_mat3x3(rot6d):
    """[N,6] -> [N,3,3] by Gram-Schmidt (transforms.py:225-234)."""
    x = rot6d.reshape(-1, 3, 2)
    a1, a2 = x[:, :, 0], x[:, :, 1]
    b1 = F.normalize(a1, dim=1)
    b2 = F.normalize(a2 - (b1 * a2).sum(-1, keepdim=True) * b1, dim=1)
    b3 = torch.cross(b1, b2, dim=1)
    return torch.stack((b1, b2, b3), dim=-1)


def rot6d_to_axis_angle(rot6d):
    """[N,6] -> [N,3] (transforms.py:197-222); NaNs (degenerate input) become 0 like the reference.
    Through the unit quaternion with Shepperd's branch selection (the largest of trace / R00 / R11 / R22 is the pivot, the
    other three components come from off-diagonal sums and differences): no cancellation for small components, stable
    near 0 and pi.  (Taking every component as sqrt(1 +- Rii ...) loses components below ~3e-4 rad: sqrt of a rounded
    difference.)  The angle is in [0, pi], torchgeometry's convention up to the sign ambiguity at exactly pi."""
    R = rot6d_to_mat3x3(rot6d)
    r00, r11, r22 = R[:, 0, 0], R[:, 1, 1], R[:, 2, 2]
    piv = torch.stack([r00 + r11 + r22, r00, r11, r22], dim=1).argmax(dim=1)
    s0 = torch.sqrt((1 + r00 + r11 + r22).clamp_min(1e-30)) * 2        # 4 w
    s1 = torch.sqrt((1 + r00 - r11 - r22).clamp_min(1e-30)) * 2        # 4 x
    s2 = torch.sqrt((1 - r00 + r11 - r22).clamp_min(1e-30)) * 2        # 4 y
    s3 = torch.sqrt((1 - r00 - r11 + r22).clamp_min(1e-30)) * 2        # 4 z
    d21, d02, d10 = R[:, 2, 1] - R[:, 1, 2], R[:, 0, 2] - R[:, 2, 0], R[:, 1, 0] - R[:, 0, 1]
    a01, a02, a12 = R[:, 0, 1] + R[:, 1, 0], R[:, 0, 2] + R[:, 2, 0], R[:, 1, 2] + R[:, 2, 1]
    cand = torch.stack([torch.stack([s0 / 4, d21 / s0, d02 / s0, d10 / s0], dim=1),
                        torch.stack([d21 / s1, s1 / 4, a01 / s1, a02 / s1], dim=1),
                        torch.stack([d02 / s2, a01 / s2, s2 / 4, a12 / s2], dim=1),
                        torch.stack([d10 / s3, a02 / s3, a12 / s3, s3 / 4], dim=1)], dim=1)      # [N, 4 branches, (w,x,y,z)]
    q = cand[torch.arange(R.shape[0], device=R.device), piv]
    q = torch.where((q[:, :1] < 0), -q, q)                              # w >= 0: angle in [0, pi]
    v = q[:, 1:]
    n = v.norm(dim=1)
    angle = 2 * torch.atan2(n, q[:, 0])
    aa = v * (angle / n.clamp_min(1e-12))[:, None]
    aa = torch.where((n < 1e-12)[:, None], 2 * v, aa)
    aa[torch.isnan(aa)] = 0.0
    return aa
