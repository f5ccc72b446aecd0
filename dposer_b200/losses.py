"""Loss, optimiser and one-step training / evaluation functions with the reference's call surface
(lib/algorithms/advanced/losses.py:31-275), running on the native training path (csrc/train.cu + csrc/gemm_tc.cu).

What differs from the reference, by construction:
  * ``loss_fn`` evaluates the loss AND (for ``train=True``) writes every parameter's gradient into ``p.grad`` in ONE
    native call -- the backward pass is hand-written, there is no autograd graph, so ``step_fn`` has no ``loss.backward()``;
  * ``get_optimizer`` returns :class:`FlatAdam`, a ``torch.optim.Adam`` subclass (same ``param_groups`` / ``state_dict``
    surface) whose parameters, gradients and moments are views into four flat buffers, so that gradient clipping + Adam
    is one kernel chain and the EMA update another;
  * the per-row time draws ``t`` come from torch's CPU generator (the schedule scalars are evaluated on the host in fp32
    like everywhere else in this package); ``z`` and the dropout masks come from Philox on the device.  All three can be
    passed in (``t=``, ``z=``, ``drop_mask=``) -- that is how the parity tests replay the reference's draws;
  * the auxiliary v2v / j2j loss ("not recommended" in the reference's config) runs as a whole inside ``step_fn``
    (:func:`auxiliary_loss_grad`): the DDIM chain keeps one native engine per network evaluation and is walked backwards
    by hand; only ``denormalize`` + the body model (a native autograd function) go through torch autograd.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L
from . import sde_lib
from . import utils as mutils
from .sde_lib import VESDE, VPSDE

_DATA_DIM = L.POSE_DIM


# ---------------------------------------------------------------------------------------------
# native engine: one dpb_train handle per (model, batch size)
# ---------------------------------------------------------------------------------------------
def _f32p(t):
    return C.cast(C.c_void_p(t.data_ptr()), L._f32p)


def _tensor_struct(model, pick):
    """dpb_train_tensors (device pointers) of the parameters (pick = lambda p: p.data) or gradients (lambda p: p.grad)."""
    w = L.ScoreWeights()

    def dp(p):
        t = pick(p)
        assert t.is_cuda and t.is_contiguous() and t.dtype == torch.float32
        return _f32p(t)
    w.pre_w, w.pre_b = dp(model.pre_dense.weight), dp(model.pre_dense.bias)
    w.pre_t_w, w.pre_t_b = dp(model.pre_dense_t.weight), dp(model.pre_dense_t.bias)
    w.pre_gn_w, w.pre_gn_b = dp(model.pre_gnorm.weight), dp(model.pre_gnorm.bias)
    w.temb_w, w.temb_b = dp(model.shared_time_embed[0].weight), dp(model.shared_time_embed[0].bias)
    names = [('b1_dense1', 'b1_gnorm1'), ('b1_dense2', 'b1_gnorm2'), ('b2_dense1', 'b2_gnorm1'), ('b2_dense2', 'b2_gnorm2')]
    for i, (dn, gn) in enumerate(names):
        w.blk_w[i], w.blk_b[i] = dp(getattr(model, dn).weight), dp(getattr(model, dn).bias)
        w.blk_t_w[i], w.blk_t_b[i] = dp(getattr(model, dn + '_t').weight), dp(getattr(model, dn + '_t').bias)
        w.blk_gn_w[i], w.blk_gn_b[i] = dp(getattr(model, gn).weight), dp(getattr(model, gn).bias)
    w.post_w, w.post_b = dp(model.post_dense.weight), dp(model.post_dense.bias)
    return w


class _Engine:
    def __init__(self, model, B, device):
        from .model import embedding_freqs
        if getattr(model, 'is_rot6d', False):
            raise NotImplementedError('the training kernels are built for the 63-D axis network, not for rot6d (126-D) '
                                      'score networks')
        if not model._geometry_ok:
            raise NotImplementedError('the training kernels are built for the shipped geometry (63-D pose, hidden 1024, '
                                      'embed 512, 2 blocks)')
        self.B, self.device = int(B), device
        self.freqs = embedding_freqs(L.EMBED).to(device=device, dtype=torch.float32).contiguous()
        out = C.c_void_p()
        L.check(L.load().dpb_train_create(C.byref(out), self.B, device.index or 0), 'dpb_train_create')
        self.ptr = out
        self.loss = torch.zeros(1, device=device)
        self.loss_rows = torch.zeros(self.B, device=device)

    def __del__(self):
        try:
            if getattr(self, 'ptr', None):
                L.load().dpb_train_destroy(self.ptr)
        except Exception:
            pass


def _engine(model, B, device):
    eng = getattr(model, '_train_engine', None)
    if eng is None or eng.B != int(B) or eng.device != device:
        eng = _Engine(model, B, device)
        model._train_engine = eng
    return eng


def native_loss(model, batch, rows, z=None, drop_mask=None, drop_p=0.0, seed=0, grads=True, clone=True, seed_dev=None):
    """One ``dpb_train_loss_grad`` call.  rows: host or device fp32 [6,B] (label, mean_c, std_c, res_c, z_c, row_w).
    Returns the loss as a [] device tensor (a fresh copy unless ``clone=False``); per-row losses stay in
    ``model._train_engine.loss_rows``."""
    L.require_cuda(batch, 'batch')
    dev = batch.device
    B = batch.shape[0]
    if batch.shape[1] != _DATA_DIM:
        raise NotImplementedError('the training kernels take the 63-D axis-angle representation')
    eng = _engine(model, B, dev)
    batch = batch.detach().to(torch.float32).contiguous()
    rows = rows.to(device=dev, dtype=torch.float32).contiguous()
    assert rows.shape == (6, B)
    P = _tensor_struct(model, lambda p: p.data)
    P.emb_freqs = _f32p(eng.freqs)
    G = None
    if grads:
        for p in model.parameters():
            if p.grad is None:
                p.grad = torch.zeros_like(p)
        G = _tensor_struct(model, lambda p: p.grad)
    if z is not None:
        z = z.to(device=dev, dtype=torch.float32).contiguous()
    if drop_mask is not None:
        drop_mask = drop_mask.to(device=dev, dtype=torch.uint8).contiguous()
        assert drop_mask.shape == (L.NUM_DENSE, B, L.HIDDEN)
    # where the Philox seed comes from: the argument, or (graph replay) device memory
    L.check(L.load().dpb_train_set_seed_pointer(eng.ptr, seed_dev))
    L.check(L.load().dpb_train_loss_grad(eng.ptr, C.byref(P), C.byref(G) if G is not None else None, L.ptr(batch),
                                         L.ptr(rows), L.ptr(z), L.ptr(drop_mask), float(drop_p), C.c_uint64(seed),
                                         L.ptr(eng.loss), L.ptr(eng.loss_rows), L.current_stream(dev)))
    return eng.loss[0].clone() if clone else eng.loss[0]


# ---------------------------------------------------------------------------------------------
# optimiser
# ---------------------------------------------------------------------------------------------
class FlatAdam(torch.optim.Adam):
    """torch.optim.Adam (amsgrad off) over flat parameter / gradient / moment buffers; ``step`` is native."""

    def __init__(self, params, lr=2e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0):
        params = list(params)
        super().__init__(params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        self._params = params
        L.require_cuda(params[0], 'parameters')
        dev = params[0].device
        n = sum(p.numel() for p in params)
        self.flat_p = torch.empty(n, device=dev)
        self.flat_g = torch.zeros(n, device=dev)
        self.flat_m = torch.zeros(n, device=dev)
        self.flat_v = torch.zeros(n, device=dev)
        self._step = 0
        self._scratch = torch.empty(int(L.load().dpb_train_adam_scratch_bytes()), dtype=torch.uint8, device=dev)
        off = 0
        with torch.no_grad():
            for p in params:
                k = p.numel()
                self.flat_p[off:off + k].copy_(p.data.reshape(-1))
                p.data = self.flat_p[off:off + k].view_as(p)
                p.grad = self.flat_g[off:off + k].view_as(p)
                off += k
        self._publish_state()

    def _views(self, flat):
        out, off = [], 0
        for p in self._params:
            out.append(flat[off:off + p.numel()].view_as(p))
            off += p.numel()
        return out

    def _publish_state(self):
        """Expose the moments through torch's per-parameter ``state`` so that ``state_dict()`` has the usual layout."""
        for p, m, v in zip(self._params, self._views(self.flat_m), self._views(self.flat_v)):
            self.state[p] = {'step': torch.tensor(float(self._step)), 'exp_avg': m, 'exp_avg_sq': v}

    def zero_grad(self, set_to_none=True):
        """Nothing to do: every gradient is overwritten by the next native backward pass (the views must stay)."""

    @torch.no_grad()
    def step(self, closure=None, grad_clip=-1.0, hyper_dev=None):
        """``hyper_dev`` (device fp32 [2], see :meth:`hyper`): the kernel reads the step size / bias correction from device
        memory -- what a captured CUDA graph of the step needs."""
        g = self.param_groups[0]
        self._step += 1
        L.check(L.load().dpb_train_adam(L.ptr(self.flat_p), L.ptr(self.flat_g), L.ptr(self.flat_m), L.ptr(self.flat_v),
                                        self.flat_p.numel(), float(g['lr']), float(g['betas'][0]), float(g['betas'][1]),
                                        float(g['eps']), float(g['weight_decay']), self._step, float(grad_clip),
                                        L.ptr(hyper_dev), L.ptr(self._scratch), L.current_stream(self.flat_p.device)))

    def _stamp(self):
        for st in self.state.values():
            st['step'] = torch.tensor(float(self._step))

    def state_dict(self):
        self._stamp()                      # the per-parameter 'step' entries are written when somebody looks
        return super().state_dict()

    def hyper(self, step):
        """(lr / (1 - beta1^step), 1 / sqrt(1 - beta2^step)) of Adam's ``step``-th update, rounded exactly like the native
        entry point does it (fp32 arguments, double arithmetic, fp32 results)."""
        g = self.param_groups[0]
        lr, b1, b2 = (float(np.float32(v)) for v in (g['lr'], g['betas'][0], g['betas'][1]))
        return float(np.float32(lr / (1.0 - b1 ** step))), float(np.float32(1.0 / np.sqrt(1.0 - b2 ** step)))

    def grad_norm(self):
        """||g||_2 over all parameters (what clip_grad_norm_ returns); synchronises."""
        L.check(L.load().dpb_train_grad_norm(L.ptr(self.flat_g), self.flat_g.numel(), L.ptr(self._scratch),
                                             L.current_stream(self.flat_g.device)))
        return float(self._scratch[:8].view(torch.float64)[0].sqrt())

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        steps = []
        with torch.no_grad():
            for p, m, v in zip(self._params, self._views(self.flat_m), self._views(self.flat_v)):
                st = self.state.get(p)
                if st:                                   # parameters torch never stepped (no gradient) have no entry
                    m.copy_(st['exp_avg'])
                    v.copy_(st['exp_avg_sq'])
                    steps.append(int(float(st['step'])))
                else:
                    m.zero_()
                    v.zero_()
        self._step = max(steps) if steps else 0
        self._publish_state()


def get_optimizer(config, params):
    """losses.py:31-41."""
    if config.optim.optimizer == 'Adam':
        return FlatAdam(params, lr=config.optim.lr, betas=(config.optim.beta1, 0.999), eps=config.optim.eps,
                        weight_decay=config.optim.weight_decay)
    raise NotImplementedError(f'Optimizer {config.optim.optimizer} not supported yet!')


def optimization_manager(config):
    """losses.py:44-57: warm-up, gradient clipping (disabled if negative), optimiser step."""

    def optimize_fn(optimizer, params, step, lr=config.optim.lr, warmup=config.optim.warmup,
                    grad_clip=config.optim.grad_clip, hyper_dev=None):
        if warmup > 0:
            for g in optimizer.param_groups:
                g['lr'] = lr * np.minimum(step / warmup, 1.0)
        optimizer.step(grad_clip=grad_clip, hyper_dev=hyper_dev)

    optimize_fn.warmup, optimize_fn.lr, optimize_fn.grad_clip = config.optim.warmup, config.optim.lr, config.optim.grad_clip
    return optimize_fn


# ---------------------------------------------------------------------------------------------
# losses
# ---------------------------------------------------------------------------------------------
def _draw_seed():
    return mutils.host_seed()


def _run(model, batch, rows, train, z, drop_mask):
    p = float(model.config.model.dropout) if train else 0.0
    loss = native_loss(model, batch, rows, z=z, drop_mask=drop_mask if train else None, drop_p=p, seed=_draw_seed(),
                       grads=train)
    return loss


def get_sde_loss_fn(sde, train, reduce_mean=False, continuous=True, likelihood_weighting=False, eps=1e-5,
                    return_data=False, denoise_steps=5):
    """losses.py:61-137.  ``loss_fn(model, batch, condition, mask, t=None, z=None, drop_mask=None)``."""
    if return_data:
        raise NotImplementedError('without autograd the estimate cannot carry gradients out of loss_fn: the auxiliary loss '
                                  'runs as a whole in get_step_fn(auxiliary_loss=True) / losses.auxiliary_loss_grad')
    red = (1.0 / _DATA_DIM) if reduce_mean else 0.5

    def make_rows(model, B, t=None):
        if t is None:
            t = torch.rand(B) * (sde.T - eps) + eps                  # losses.py:111 (CPU generator here)
        t = t.detach().to('cpu', torch.float32)
        # labels, score multiplier m (score = m * res), marginal mean coefficient and std: the samplers' table helper
        coef, labels = mutils.em_coefficients(sde, model, t, probability_flow=True, continuous=continuous)
        m, mean_c, std = coef[:, 5], coef[:, 3], coef[:, 4]
        if not likelihood_weighting:
            res_c, z_c, w = m * std, torch.ones(B), torch.full((B,), red)           # (score std + z)^2
        else:
            g2 = sde.sde(torch.zeros(B, 1), t)[1] ** 2
            res_c, z_c, w = m, 1.0 / std, red * g2                                  # (score + z / std)^2 g^2
        return torch.stack([labels.float(), mean_c, std, res_c, z_c, w])

    def loss_fn(model, batch, condition=None, mask=None, t=None, z=None, drop_mask=None):
        return _run(model, batch, make_rows(model, batch.shape[0], t), train, z, drop_mask)

    loss_fn.make_rows = make_rows
    return loss_fn


def get_smld_loss_fn(vesde, train, reduce_mean=False):
    """losses.py:140-161 (legacy NCSN objective; labels index the DESCENDING sigma array)."""
    assert isinstance(vesde, VESDE), "SMLD training only works for VESDEs."
    smld_sigma_array = torch.flip(vesde.discrete_sigmas, dims=(0,))
    red = (1.0 / _DATA_DIM) if reduce_mean else 0.5

    def make_rows(model, B, labels=None):
        if labels is None:
            labels = torch.randint(0, vesde.N, (B,))
        labels = labels.cpu()
        sig = smld_sigma_array[labels]
        inv_s = 1.0 / mutils.sigma_at(model, labels.float())
        # score = res / sigmas[label]; target = -z / sig; (score - target)^2 sig^2
        return torch.stack([labels.float(), torch.ones(B), sig, inv_s, 1.0 / sig, red * sig ** 2])

    def loss_fn(model, batch, condition=None, mask=None, labels=None, z=None, drop_mask=None):
        return _run(model, batch, make_rows(model, batch.shape[0], labels), train, z, drop_mask)

    loss_fn.make_rows = make_rows
    return loss_fn


def get_ddpm_loss_fn(vpsde, train, reduce_mean=True):
    """losses.py:164-184 (legacy DDPM objective)."""
    assert isinstance(vpsde, VPSDE), "DDPM training only works for VPSDEs."
    red = (1.0 / _DATA_DIM) if reduce_mean else 0.5

    def make_rows(model, B, labels=None):
        if labels is None:
            labels = torch.randint(0, vpsde.N, (B,))
        labels = labels.cpu()
        inv_s = 1.0 / mutils.sigma_at(model, labels.float())
        return torch.stack([labels.float(), vpsde.sqrt_alphas_cumprod[labels], vpsde.sqrt_1m_alphas_cumprod[labels],
                            inv_s, -torch.ones(B), torch.full((B,), red)])            # (score - noise)^2

    def loss_fn(model, batch, condition=None, mask=None, labels=None, z=None, drop_mask=None):
        return _run(model, batch, make_rows(model, batch.shape[0], labels), train, z, drop_mask)

    loss_fn.make_rows = make_rows
    return loss_fn


# ---------------------------------------------------------------------------------------------
# auxiliary loss: DDIM chain under the optimiser + body model (losses.py:91-106,117-121,244-258)
# ---------------------------------------------------------------------------------------------
def _rows_axpby(a, x, b=None, y=None):
    """out[r,c] = a[r] x[r,c] (+ b[r] y[r,c]) -- native, device fp32."""
    out = torch.empty_like(x)
    L.check(L.load().dpb_rows_axpby(L.ptr(a), L.ptr(x), L.ptr(b), L.ptr(y), L.ptr(out), x.shape[1], x.shape[0],
                                    L.current_stream(x.device)))
    return out


def _weighted_sqdiff(p, q, w, scale, want_grad=True):
    """(scale * sum_b w[b] sum (p - q)^2 as a [1] tensor, d/dq or None) -- native."""
    B = p.shape[0]
    n = p[0].numel()
    loss = torch.empty(1, device=p.device)
    grad = torch.empty_like(q) if want_grad else None
    scratch = torch.empty(B, device=p.device)
    L.check(L.load().dpb_weighted_sqdiff(L.ptr(p), L.ptr(q), L.ptr(w), B, n, float(scale), L.ptr(loss), L.ptr(grad),
                                         L.ptr(scratch), L.current_stream(p.device)))
    return loss, grad


def auxiliary_loss_grad(model, sde, batch, denormalize, body_model, denoise_steps=5, reduce_mean=False, continuous=True,
                        eps=1e-5, t=None, z=None, drop_mask=None, score_scale=1.0):
    """Loss of get_step_fn(auxiliary_loss=True) (losses.py:244-258) and every parameter gradient, without autograd through
    the network: ``denoise_steps`` network evaluations of multi_step_denoise (each on its own native engine, activations
    kept), the estimate through ``denormalize`` + ``body_model`` (torch autograd over the native LBS function), weighted
    v2v / j2j terms, then the chain backwards -- every evaluation's backward adds into the same flat gradient buffers.
    ``drop_mask``: [denoise_steps, 5, B, 1024] keep-masks (parity mode); ``score_scale`` multiplies the score-matching term
    (tests switch it off to look at the body-model terms alone).  Returns a dict of [] device tensors."""
    from .misc import linear_interpolation
    L.require_cuda(batch, 'batch')
    lib = L.load()
    dev, B, N = batch.device, batch.shape[0], int(denoise_steps)
    st = L.current_stream(dev)
    p_drop = float(model.config.model.dropout)
    engines = getattr(model, '_aux_engines', None)
    if engines is None or len(engines) != N or engines[0].B != B or engines[0].device != dev:
        engines = model._aux_engines = [_Engine(model, B, dev) for _ in range(N)]
    for prm in model.parameters():
        if prm.grad is None:
            prm.grad = torch.zeros_like(prm)
    P = _tensor_struct(model, lambda q: q.data)
    P.emb_freqs = _f32p(engines[0].freqs)
    G = _tensor_struct(model, lambda q: q.grad)
    up = lambda v: v.to(device=dev, dtype=torch.float32).contiguous()                 # noqa: E731
    # ---- host scalars of the chain (fp32 torch expressions of the reference)
    if t is None:
        t = torch.rand(B) * (sde.T - eps) + eps
    t = t.detach().to('cpu', torch.float32)
    traj = linear_interpolation(t, t / (2 * N), N + 1)                                 # losses.py:92,120
    coef0, _ = mutils.em_coefficients(sde, model, t, probability_flow=True, continuous=continuous)
    mean_c, std0, m0 = coef0[:, 3], coef0[:, 4], coef0[:, 5]
    alpha0, sigma0 = sde.return_alpha_sigma(t)
    weight = torch.log(1.0 + alpha0[:, 0] / sigma0)                                    # log(1 + SNR), losses.py:246
    labels, c1s, c2s = [], [], []
    for i in range(N):
        tc, tb = traj[i], traj[i + 1]
        a_c, s_c = sde.return_alpha_sigma(tc)
        a_b, s_b = sde.return_alpha_sigma(tb)
        cf, lab = mutils.em_coefficients(sde, model, tc, probability_flow=True, continuous=continuous)
        c1 = (a_b / a_c)[:, 0]
        labels.append(up(lab))
        c1s.append(up(c1))
        c2s.append(up(-(s_b - c1 * s_c) * cf[:, 5] * s_c))          # x' = c1 x + (s_b - c1 s_c) noise, noise = -m res s_c
    ones = torch.ones(B, device=dev)
    # ---- forward chain
    batch = batch.detach().to(torch.float32).contiguous()
    if z is None:
        z = torch.empty(B, _DATA_DIM, device=dev)
        L.check(lib.dpb_normal_fill(L.ptr(z), B, C.c_uint64(_draw_seed()), C.c_uint64(0), 0, st))
    else:
        z = up(z)
    x = _rows_axpby(up(mean_c), batch, up(std0), z)                                    # perturbed data, losses.py:113-115
    seeds = [_draw_seed() for _ in range(N)]
    masks = [None] * N if drop_mask is None else [drop_mask[i].to(device=dev, dtype=torch.uint8).contiguous() for i in range(N)]
    res0 = None
    for i in range(N):
        res = torch.empty(B, _DATA_DIM, device=dev)
        L.check(lib.dpb_train_forward(engines[i].ptr, C.byref(P), L.ptr(x), L.ptr(labels[i]), L.ptr(masks[i]), p_drop,
                                      C.c_uint64(seeds[i]), L.ptr(res), st))
        if i == 0:
            res0 = res
        x = _rows_axpby(c1s[i], x, c2s[i], res)
    # ---- score-matching term on the first evaluation: (score std + z)^2 = rc^2 (res - (-z / rc))^2, rc = m std
    red = (1.0 / _DATA_DIM) if reduce_mean else 0.5
    rc = m0 * std0
    target = _rows_axpby(up(-1.0 / rc), z)
    score_loss, g_res_score = _weighted_sqdiff(target, res0, up(red * rc * rc), float(score_scale) / B)
    # ---- body-model terms on the estimate (torch autograd over denormalize + the native LBS function)
    wdev = up(weight)
    with torch.no_grad():                      # the target first: the body model keeps ONE saved forward state per module
        gt = body_model(pose_body=denormalize(batch))
        gt_v, gt_j = gt.v.clone(), gt.Jtr.clone()
    with torch.enable_grad():
        leaf = x.detach().requires_grad_(True)
        pred = body_model(pose_body=denormalize(leaf))
        loss_v2v, g_v = _weighted_sqdiff(gt_v, pred.v.detach().contiguous(), wdev, 1.0 / (B * pred.v.shape[1]))
        loss_j2j, g_j = _weighted_sqdiff(gt_j, pred.Jtr.detach().contiguous(), wdev, 1.0 / (B * pred.Jtr.shape[1]))
        torch.autograd.backward([pred.v, pred.Jtr], [g_v.view_as(pred.v), g_j.view_as(pred.Jtr)])
    g_x = leaf.grad.contiguous()
    # ---- chain backwards: the first call overwrites the gradients, the others add
    for i in reversed(range(N)):
        g_res = _rows_axpby(c2s[i], g_x, ones, g_res_score) if i == 0 else _rows_axpby(c2s[i], g_x)
        g_in = torch.empty(B, _DATA_DIM, device=dev) if i > 0 else None
        L.check(lib.dpb_train_backward(engines[i].ptr, C.byref(P), C.byref(G), L.ptr(g_res), L.ptr(masks[i]), p_drop,
                                       C.c_uint64(seeds[i]), 0 if i == N - 1 else 1, L.ptr(g_in), st))
        if i > 0:
            g_x = _rows_axpby(c1s[i], g_x, ones, g_in)
    loss = score_loss + loss_v2v + loss_j2j
    return {'step_loss': loss[0], 'score_loss': score_loss[0], 'v2v_loss': loss_v2v[0], 'j2j_loss': loss_j2j[0]}


class _GraphedStep:
    """loss + backward + clip + Adam + EMA of one batch size as ONE captured CUDA graph.  What changes from step to step --
    the per-row schedule scalars, the Philox seed, Adam's step size / bias correction, the EMA decay -- lives in one
    device buffer that a single small host-to-device copy refreshes before every replay."""

    def __init__(self, model, optimizer, ema, B, dev, grad_clip):
        self.B, self.dev = B, dev
        self.eng = _engine(model, B, dev)
        self.buf = torch.zeros(8 + 6 * B, device=dev)            # [step_size, inv_sqrt_bc2, omd, -, seed lo, seed hi, -, -, rows]
        self.host = torch.zeros(8 + 6 * B)
        self.batch = torch.zeros(B, _DATA_DIM, device=dev)
        rows, hyper = self.buf[8:].view(6, B), self.buf[:3]
        seed_dev = C.c_void_p(self.buf.data_ptr() + 16)
        p = float(model.config.model.dropout)
        keep = (optimizer._step, ema.num_updates)

        def body():
            native_loss(model, self.batch, rows, drop_p=p, seed=0, grads=True, clone=False, seed_dev=seed_dev)
            optimizer.step(grad_clip=grad_clip, hyper_dev=hyper[:2])
            ema.update(model.parameters(), omd_dev=hyper[2:])
        self.graph = torch.cuda.CUDAGraph()
        torch.cuda.synchronize(dev)
        with torch.cuda.graph(self.graph):
            body()
        optimizer._step, ema.num_updates = keep                  # capture launched nothing: undo the host-side counters

    def run(self, optimizer, ema, batch, rows, lr_t):
        for g in optimizer.param_groups:
            g['lr'] = lr_t
        optimizer._step += 1
        h = self.host
        h[0], h[1] = optimizer.hyper(optimizer._step)
        h[2] = ema.next_one_minus_decay()
        h[4:6] = torch.tensor([_draw_seed()], dtype=torch.int64).view(torch.float32)
        h[8:] = rows.reshape(-1)
        self.buf.copy_(h)                                        # pageable source: the copy is complete when this returns
        self.batch.copy_(batch, non_blocking=True)
        self.graph.replay()
        if ema.num_updates is not None:
            ema.num_updates += 1
        return self.eng.loss[0].clone()


def get_step_fn(sde, train, optimize_fn=None, reduce_mean=False, continuous=True, likelihood_weighting=False,
                auxiliary_loss=False, denormalize=None, body_model=None, rot_rep='rot6d', denoise_steps=5, graph=False,
                data_parallel=False):
    """losses.py:187-275: ``step_fn(state, batch)`` with ``state = dict(optimizer, model, ema, step)``.
    ``graph=True``: the training step of each batch size is captured once as a CUDA graph and replayed (needs the
    optimize_fn of :func:`optimization_manager`; steps that replay given draws -- ``z=`` / ``drop_mask=`` -- run eagerly).
    ``data_parallel=True`` (one process per GPU, ``torch.distributed`` initialised): every rank steps on its own shard of the
    batch and the flat gradient buffer is averaged over ranks with ONE all-reduce before clipping / Adam -- the reference
    trains on one GPU (run/train.py), this is the collective SURVEY 8(e)/(f)3 names for scaling it out."""
    from . import dist as D
    if auxiliary_loss:
        assert denormalize is not None and body_model is not None
        if rot_rep != 'axis':
            raise NotImplementedError("the auxiliary loss is built for rot_rep='axis' (the 63-D network input)")
        if not continuous or likelihood_weighting:
            raise NotImplementedError('the auxiliary loss goes with the continuous, unweighted SDE loss')
    if continuous:
        loss_fn = get_sde_loss_fn(sde, train, reduce_mean=reduce_mean, continuous=True,
                                  likelihood_weighting=likelihood_weighting)
    else:
        assert not likelihood_weighting, "Likelihood weighting is not supported for original SMLD/DDPM training."
        if isinstance(sde, VESDE):
            loss_fn = get_smld_loss_fn(sde, train, reduce_mean=reduce_mean)
        elif isinstance(sde, VPSDE):
            loss_fn = get_ddpm_loss_fn(sde, train, reduce_mean=reduce_mean)
        else:
            raise ValueError(f"Discrete training for {sde.__class__.__name__} is not recommended.")

    graphs = {}

    def step_fn(state, batch, condition=None, mask=None, **draws):
        model = state['model']
        if train and graph and not data_parallel and not auxiliary_loss and 'z' not in draws and 'drop_mask' not in draws:
            optimizer, ema, B = state['optimizer'], state['ema'], batch.shape[0]
            L.require_cuda(batch, 'batch')
            g = graphs.get(B)
            if g is None:
                g = graphs[B] = _GraphedStep(model, optimizer, ema, B, batch.device, optimize_fn.grad_clip)
            rows = loss_fn.make_rows(model, B, **draws)
            warm, lr = optimize_fn.warmup, optimize_fn.lr
            lr_t = lr * min(state['step'] / warm, 1.0) if warm > 0 else lr
            loss = g.run(optimizer, ema, batch.detach().to(torch.float32), rows, lr_t)
            state['step'] += 1
            model.mark_updated()
        elif train and auxiliary_loss:
            optimizer = state['optimizer']
            ld = auxiliary_loss_grad(model, sde, batch, denormalize, body_model, denoise_steps=denoise_steps,
                                     reduce_mean=reduce_mean, **draws)
            if data_parallel:
                D.all_reduce_mean_(optimizer.flat_g)
            optimize_fn(optimizer, model.parameters(), step=state['step'])
            state['step'] += 1
            model.mark_updated()
            state['ema'].update(model.parameters())
            return ld
        elif train:
            optimizer = state['optimizer']
            optimizer.zero_grad()
            loss = loss_fn(model, batch, condition, mask, **draws)       # loss and every p.grad in one native call
            if data_parallel:
                D.all_reduce_mean_(optimizer.flat_g)
            optimize_fn(optimizer, model.parameters(), step=state['step'])
            state['step'] += 1
            model.mark_updated()
            state['ema'].update(model.parameters())
        else:
            with torch.no_grad():
                ema = state['ema']
                ema.store(model.parameters())
                ema.copy_to(model.parameters())
                loss = loss_fn(model, batch, condition, mask, **draws)
                ema.restore(model.parameters())
        return {'step_loss': loss, 'score_loss': loss}

    return step_fn
