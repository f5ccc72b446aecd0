"""DPoser prior loss with the reference's call surface.

Replaces ``DPoserComp`` (run/completion.py:95-207), ``MotionDenoise.DPoser_loss``
(run/motion_denoising.py:125-143) and ``DPoser`` (run/smplify.py:17-115).  One call into
``dpb_prior_loss`` does perturb -> score net -> one-step denoise -> weighted squared error
and its closed-form gradient (x0_hat is detached in the reference, so no backward through
the network exists).  The returned loss is an autograd scalar whose backward scales the
kernel-produced gradient.
"""
import math

import torch
import torch.nn as nn

from . import _lib as L
from . import utils as mutils
from .misc import linear_interpolation

N_POSES = 21


class _PriorLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x0, owner, t, weighted, divisor, z, seed):
        model = owner.model
        ps = mutils.prior_scalars(owner.sde, model, t, owner.continuous)
        table = owner._table(t, ps['label'])
        xd = x0.detach().to(torch.float32).contiguous()
        L.require_cuda(xd, 'x_0')
        B = xd.shape[0]
        loss = torch.empty(1, dtype=torch.float32, device=xd.device)
        grad = torch.empty_like(xd)
        h = model.handle()
        ws = model.workspace(B, xd.device)
        zz = None if z is None else z.detach().to(torch.float32).contiguous()
        L.check(L.load().dpb_prior_loss(h.ptr, L.ptr(xd), L.ptr(table), ps['alpha'], ps['std'], ps['inv_sigma_std'],
                                        int(bool(weighted)), float(divisor), L.ptr(zz), seed, 0, L.ptr(loss),
                                        L.ptr(grad), None, B, model.engine, L.ptr(ws), ws.numel(),
                                        L.current_stream(xd.device)))
        ctx.save_for_backward(grad)
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        (grad,) = ctx.saved_tensors
        return grad * g, None, None, None, None, None, None


class _PriorBase:
    """Shared machinery: cached per-t time tables and the fused loss call."""

    def _init_prior(self, model, sde, continuous, batch_size):
        self.model, self.sde, self.continuous, self.batch_size = model, sde, continuous, batch_size
        self.score_fn = mutils.get_score_fn(sde, model, train=False, continuous=continuous)
        self.rsde = sde.reverse(self.score_fn, False)
        self.loss_fn = nn.MSELoss(reduction='none')
        self._tables = {}

    def _table(self, t, label):
        # the tables are built from the handle's weights: a weight reload / device move gives a new handle
        # (ScoreModelFC.handle()), and every cached table is dropped with the old one
        h = self.model.handle()
        if getattr(self, '_tables_handle', None) is not h:
            self._tables, self._tables_handle = {}, h
        key = float(t)
        tb = self._tables.get(key)
        if tb is None:
            tb = self.model.time_table(label)
            self._tables[key] = tb
        return tb

    @staticmethod
    def _host_t(vec_t):
        """The batch-uniform time as a python float (one tiny D2H read when given a device tensor)."""
        if isinstance(vec_t, (float, int)):
            return float(vec_t)
        return float(vec_t.reshape(-1)[0])

    def _fused_loss(self, x_0, t, weighted, divisor, z=None):
        self.model.check_width(x_0, 'x_0')
        if z is not None:
            self.model.check_width(z, 'z', x_0.shape[0])
        seed = mutils.host_seed() if z is None else 0
        return _PriorLossFn.apply(x_0, self, t, weighted, divisor, z, seed)

    # the un-fused pieces keep the reference's names for callers that use them directly
    def one_step_denoise(self, x_t, t):
        """run/completion.py:105-110."""
        drift, diffusion, alpha, sigma_2, score = self.rsde.sde(x_t, t, guide=True)
        x_0_hat = (x_t.detach() + sigma_2[:, None] * score) / alpha
        return x_0_hat.detach(), alpha / torch.sqrt(sigma_2)[:, None]

    def multi_step_denoise(self, x_t, t, t_end, N=10):
        """run/completion.py:112-129 (DDIM).  Every DDIM step is affine in (x, raw network output):
            x' = (a_b / a_c) x + [s_c (s_b - s_c a_b / a_c) / (sigma std)] raw
        so the N steps are ONE ``dpb_sampler_run`` with an N-row coefficient table (noise coefficient 0): with the tcgen05
        engine a single persistent kernel, like the reverse-SDE sampler."""
        from . import sampling
        self.model.check_width(x_t, 'x_t')
        t0, t1 = self._host_t(t), self._host_t(t_end)
        traj = torch.linspace(0, 1, N + 1)
        traj = (1 - traj) * t0 + traj * t1                      # linear_interpolation (lib/utils/misc.py:58-61)
        coef = torch.zeros(N, L.COEF_STRIDE)
        labels = []
        for i in range(N):
            tc, tb = traj[i:i + 1].float(), traj[i + 1:i + 2].float()
            a_c, s_c = self.sde.return_alpha_sigma(tc)
            a_b, s_b = self.sde.return_alpha_sigma(tb)
            ps = mutils.prior_scalars(self.sde, self.model, float(tc), self.continuous)
            ratio = (a_b / a_c).reshape(-1)[0]
            coef[i, 0] = ratio
            coef[i, 1] = s_c.reshape(-1)[0] * ps['inv_sigma_std'] * (s_b.reshape(-1)[0] - s_c.reshape(-1)[0] * ratio)
            coef[i, 3], coef[i, 4] = 1.0, 0.0
            labels.append(ps['label'])
        cur = x_t.detach().to(torch.float32).contiguous().clone()
        L.require_cuda(cur, 'x_t')
        table = self.model.time_table(torch.cat(labels))
        x_mean = torch.empty_like(cur)
        sampling._run_steps(self.model, cur, coef.to(cur.device), table, None, None, None, 0, 0, None, x_mean, False)
        alpha, sigma = self.sde.return_alpha_sigma(torch.tensor([t0], dtype=torch.float32))
        snr = (alpha.reshape(-1)[0] / sigma.reshape(-1)[0]).to(cur.device).expand(cur.shape[0], 1)
        return x_mean, snr

    def _ddim_loss(self, x_0, vec_t, weighted, divisor, n, z=None):
        """multi_denoise=True branch: only the final squared error is differentiable w.r.t. x_0."""
        self.model.check_width(x_0, 'x_0')
        if z is not None:
            self.model.check_width(z, 'z', x_0.shape[0])
        z = torch.randn_like(x_0) if z is None else z
        mean, std = self.sde.marginal_prob(x_0, vec_t)
        x0_hat, snr = self.multi_step_denoise(mean + std[:, None] * z, vec_t, t_end=vec_t / (2 * n), N=n)
        w = 0.5 * torch.sqrt(1 + snr) if weighted else 0.5
        sq = w * self.loss_fn(x_0, x0_hat)
        return sq.mean() if divisor is None else sq.sum() / divisor


class DPoserComp(_PriorBase):
    """run/completion.py:95-207."""

    def __init__(self, diffusion_model, sde, continuous, batch_size=1):
        self._init_prior(diffusion_model, sde, continuous, batch_size)
        self.data_loss = nn.MSELoss(reduction='mean')

    def loss(self, x_0, vec_t, weighted=False, multi_denoise=False, z=None):
        """mean over B*D of w (x0 - sg[x0_hat])^2  (run/completion.py:131-149)."""
        if multi_denoise:
            return self._ddim_loss(x_0, vec_t, weighted, None, 10, z)
        return self._fused_loss(x_0, self._host_t(vec_t), bool(weighted), float(x_0.numel()), z)

    def get_loss_weights(self):
        return {'data': lambda cst, it: 100 * cst / (1 + it), 'dposer': lambda cst, it: 0.1 * cst * (it + 1)}

    @staticmethod
    def backward_step(loss_dict, weight_dict, it):
        return torch.stack([weight_dict[k](loss_dict[k], it) for k in loss_dict]).sum()

    def optimize(self, observation, mask, time_strategy='3', lr=0.1, sample_trun=5.0, sample_time=900,
                 iterations=2, steps_per_iter=100, z_list=None, graphs=False):
        """run/completion.py:167-207: Adam on the pose with data + DPoser losses.  Per step three kernels: prior loss
        with its closed-form gradient, the masked-MSE cotangent, fused Adam (no framework op, no autograd).
        ``z_list`` (parity mode): the Gaussian draw of every step; ``graphs``: capture / replay every step as a CUDA graph."""
        from . import steps as S
        self.model.check_width(observation, 'observation')
        if mask.shape[-1] != self.model.pose_width:
            raise ValueError(f'mask: expected its last dimension to be {self.model.pose_width}, got {list(mask.shape)}')
        if z_list is not None:
            for z in z_list:
                self.model.check_width(z, 'z_list entry', observation.shape[0])
        L.require_cuda(observation, 'observation')
        dev = observation.device
        total_steps = iterations * steps_per_iter
        obs = observation.detach().to(torch.float32).contiguous()
        msk = mask.detach().to(torch.float32).expand_as(obs).contiguous()
        x = obs.clone()
        rows = x.shape[0]
        timesteps = mutils.timestep_grid(self.sde, 1e-3)           # host copy: no per-step device read
        sched = []
        for it in range(iterations):
            for i in range(steps_per_iter):
                step = it * steps_per_iter + i
                if time_strategy == '1':
                    quan_t = int(torch.randint(self.sde.N, [1]))
                elif time_strategy == '2':
                    quan_t = int(sample_time)
                elif time_strategy == '3':
                    quan_t = self.sde.N - math.floor(
                        torch.tensor(total_steps - step - 1) * (self.sde.N / (sample_trun * total_steps))) - 2
                else:
                    raise NotImplementedError('unsupported time sampling strategy')
                sched.append((it, quan_t, float(timesteps[quan_t])))
        pri = S.PriorStep(self.model, self.sde, self.continuous, rows, dev)
        pri.schedule([t for _, _, t in sched])
        g_data = torch.empty_like(x)
        zbuf = torch.empty_like(x) if z_list is not None else None
        D = self.model.pose_width
        opt = S.Adam(x, 0, D, lr)
        wd = self.get_loss_weights()
        seed = mutils.host_seed() if z_list is None else 0
        sg = S.StepGraphs(graphs and z_list is None)
        lib = L.load()

        def one_step(k):
            it, quan_t, _ = sched[k]
            z = None
            if z_list is not None:
                zbuf.copy_(z_list[k].to(dev))
                z = zbuf
            # the reference passes quan_t into `weighted` (run/completion.py:196): weighted iff quan_t != 0
            pri(x, k, bool(quan_t), float(x.numel()), z=z, seed=seed, step=k)
            L.check(lib.dpb_masked_mse_grad(L.ptr(x), L.ptr(obs), L.ptr(msk), L.ptr(g_data), x.numel(),
                                            L.current_stream(dev)))
            opt.step(g_data, 0, D, wd['data'](1.0, it), g2=pri.grad, off2=0, ld2=D, s2=wd['dposer'](1.0, it))

        for k in range(total_steps):
            sg.run(k, lambda k=k: one_step(k))
        return obs * msk + x * (1.0 - msk)


class MotionPrior(_PriorBase):
    """The prior part of ``MotionDenoise`` (run/motion_denoising.py:63-143)."""

    def __init__(self, diffusion_model, sde, continuous=True, batch_size=1):
        self._init_prior(diffusion_model, sde, continuous, batch_size)

    def DPoser_loss(self, x_0, vec_t, quan_t=None, weighted=False, multi_denoise=False, z=None):
        """sum_all(w (x0 - sg[x0_hat])^2) / batch_size  (run/motion_denoising.py:125-143)."""
        if multi_denoise:
            return self._ddim_loss(x_0, vec_t, weighted, self.batch_size, 10, z)
        return self._fused_loss(x_0, self._host_t(vec_t), bool(weighted), float(self.batch_size), z)


class DPoser(nn.Module, _PriorBase):
    """run/smplify.py:17-115 -- SMPLify pose prior: normalise, weighted loss, sum / batch_size."""

    def __init__(self, batch_size=32, config_path='', args=None, model=None, sde=None, normalizer=None,
                 continuous=True):
        nn.Module.__init__(self)
        if model is None or sde is None or normalizer is None:
            raise NotImplementedError('checkpoint / config loading is out of scope: pass model=, sde=, normalizer=')
        self.device = getattr(args, 'device', None)
        self.Normalizer = normalizer
        sde.N = getattr(args, 'sde_N', sde.N)
        self._init_prior(model, sde, continuous, batch_size)
        self.timesteps = mutils.timestep_grid(sde, 1e-3)

    def DPoser_loss(self, x_0, vec_t, multi_denoise=False, z=None):
        if multi_denoise:
            return self._ddim_loss(x_0, vec_t, True, self.batch_size, 5, z)
        return self._fused_loss(x_0, self._host_t(vec_t), True, float(self.batch_size), z)

    def forward(self, poses, betas, quan_t):
        poses = self.Normalizer.offline_normalize(poses[:, :N_POSES * 3], from_axis=True)
        return self.DPoser_loss(poses, float(self.timesteps[int(quan_t)]))
