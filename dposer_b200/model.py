"""Drop-in ``ScoreModelFC`` (reference lib/algorithms/advanced/model.py:93-196).

Same constructor, same parameter / buffer names (``state_dict`` compatible, including the
unused ``pre_dense_cond``), same ``forward(batch, t, condition=None, mask=None)``.  The
forward pass runs in libdposer_b200: the time path (sinusoidal embedding, shared embed,
five ``*_t`` projections) is evaluated once per distinct label and the x-path runs either on
the tcgen05 engine (batch-uniform t) or on the fp32 engine.

Not differentiable: every hot-path caller detaches the network output
(run/completion.py:109, run/motion_denoising.py:103, run/smplify.py:73); backward through the
net is a "next" row (SURVEY 8f).
"""
import ctypes as C
import math

import numpy as np
import torch
import torch.nn as nn

from . import _lib as L


def get_sigmas(config):
    """model.py:24-34 -- exp(linspace(log sigma_max, log sigma_min, num_scales)) (numpy fp64)."""
    return np.exp(np.linspace(np.log(config.model.sigma_max), np.log(config.model.sigma_min),
                              config.model.num_scales))


def embedding_freqs(embedding_dim, max_positions=10000):
    """The fp32 frequency vector of model.py:41-43, evaluated with the same torch expression."""
    half = embedding_dim // 2
    scale = math.log(max_positions) / (half - 1)
    return torch.exp(torch.arange(half, dtype=torch.float32) * -scale)


def get_act(config):
    """model.py:54-66.  Only swish is wired into the kernels."""
    name = config.model.nonlinearity.lower()
    if name == 'swish':
        return nn.SiLU()
    if name in ('elu', 'relu', 'lrelu'):
        raise NotImplementedError(f'activation {name!r} is not built into the B200 kernels (swish only)')
    raise NotImplementedError('activation function does not exist!')


class _Handle:
    """Owns a dpb_score_t* and the parameter versions it was built from."""

    def __init__(self, ptr, device, versions):
        self.ptr, self.device, self.versions = ptr, device, versions

    def __del__(self):
        try:
            if self.ptr:
                L.load().dpb_score_destroy(self.ptr)
        except Exception:
            pass


class ScoreModelFC(nn.Module):
    def __init__(self, config, n_poses=21, pose_dim=6, hidden_dim=64, embed_dim=32, n_blocks=2):
        super().__init__()
        self.config = config
        self.n_poses = n_poses
        self.joint_dim = pose_dim
        self.n_blocks = n_blocks
        self.act = get_act(config)
        # identical registration order to the reference so torch.manual_seed(s) gives identical weights
        self.pre_dense = nn.Linear(n_poses * pose_dim, hidden_dim)
        self.pre_dense_t = nn.Linear(embed_dim, hidden_dim)
        self.pre_dense_cond = nn.Linear(hidden_dim, hidden_dim)   # constructed but unused (model.py:111)
        self.pre_gnorm = nn.GroupNorm(32, num_channels=hidden_dim)
        self.dropout = nn.Dropout(p=config.model.dropout)
        self.time_embedding_type = config.model.embedding_type.lower()
        if self.time_embedding_type != 'positional':
            raise NotImplementedError("only embedding_type='positional' is built (the shipped config)")
        self.shared_time_embed = nn.Sequential(nn.Linear(embed_dim, embed_dim), self.act)
        self.register_buffer('sigmas', torch.tensor(get_sigmas(config), dtype=torch.float))
        for idx in range(n_blocks):
            setattr(self, f'b{idx + 1}_dense1', nn.Linear(hidden_dim, hidden_dim))
            setattr(self, f'b{idx + 1}_dense1_t', nn.Linear(embed_dim, hidden_dim))
            setattr(self, f'b{idx + 1}_gnorm1', nn.GroupNorm(32, num_channels=hidden_dim))
            setattr(self, f'b{idx + 1}_dense2', nn.Linear(hidden_dim, hidden_dim))
            setattr(self, f'b{idx + 1}_dense2_t', nn.Linear(embed_dim, hidden_dim))
            setattr(self, f'b{idx + 1}_gnorm2', nn.GroupNorm(32, num_channels=hidden_dim))
        self.post_dense = nn.Linear(hidden_dim, n_poses * pose_dim)
        # input / output width D: 63 (axis-angle, pose_dim=3) or 126 (rot6d, pose_dim=6)
        self.pose_width = n_poses * pose_dim
        self._geometry_ok = (self.pose_width in L.POSE_DIMS and hidden_dim == L.HIDDEN and
                             embed_dim == L.EMBED and n_blocks == 2)
        self._h = None
        self._ws = {}
        self._native_updates = 0
        self.engine = L.ENGINE_AUTO      # ENGINE_FP32 forces the exact path, ENGINE_TC the tensor-core path

    # ------------------------------------------------------------------ handle management
    def _param_versions(self):
        return (self._native_updates,) + tuple((p.data_ptr(), p._version) for p in self.parameters())

    def mark_updated(self):
        """The native optimiser wrote the weights in place (no torch version bump): rebuild the handle on next use."""
        self._native_updates += 1

    def handle(self):
        """Create (or refresh after a weight update) the device handle built from the current weights."""
        dev = self.pre_dense.weight.device
        if dev.type != 'cuda':
            raise RuntimeError('dposer_b200.ScoreModelFC runs on CUDA only (no CPU fallback): call .cuda() first')
        if not self._geometry_ok:
            raise NotImplementedError('kernels are built for the shipped geometry: 63-D (axis) or 126-D (rot6d) pose, '
                                      'hidden 1024, embed 512, 2 blocks (configs/subvp/amass_scorefc_continuous.py)')
        ver = self._param_versions()
        if self._h is not None and self._h.versions == ver:
            return self._h
        lib = L.load()
        w = L.ScoreWeights()
        keep = []

        def hp(t):
            a, p = L.host_f32(t)
            keep.append(a)
            return p
        w.pre_w, w.pre_b = hp(self.pre_dense.weight), hp(self.pre_dense.bias)
        w.pre_t_w, w.pre_t_b = hp(self.pre_dense_t.weight), hp(self.pre_dense_t.bias)
        w.pre_gn_w, w.pre_gn_b = hp(self.pre_gnorm.weight), hp(self.pre_gnorm.bias)
        w.temb_w, w.temb_b = hp(self.shared_time_embed[0].weight), hp(self.shared_time_embed[0].bias)
        names = [('b1_dense1', 'b1_gnorm1'), ('b1_dense2', 'b1_gnorm2'), ('b2_dense1', 'b2_gnorm1'),
                 ('b2_dense2', 'b2_gnorm2')]
        for i, (dn, gn) in enumerate(names):
            w.blk_w[i], w.blk_b[i] = hp(getattr(self, dn).weight), hp(getattr(self, dn).bias)
            w.blk_t_w[i], w.blk_t_b[i] = hp(getattr(self, dn + '_t').weight), hp(getattr(self, dn + '_t').bias)
            w.blk_gn_w[i], w.blk_gn_b[i] = hp(getattr(self, gn).weight), hp(getattr(self, gn).bias)
        w.post_w, w.post_b = hp(self.post_dense.weight), hp(self.post_dense.bias)
        w.emb_freqs = hp(embedding_freqs(L.EMBED))
        out = C.c_void_p()
        L.check(lib.dpb_score_create_dim(C.byref(out), C.byref(w), self.pose_width, dev.index or 0), 'dpb_score_create_dim')
        self._h = _Handle(out, dev, ver)
        return self._h

    def workspace(self, B, device):
        """Caller-owned scratch for the fp32 engine, cached per batch size."""
        key = (int(B), str(device))
        ws = self._ws.get(key)
        if ws is None:
            n = L.load().dpb_score_workspace_bytes(self.handle().ptr, int(B), 0)
            ws = torch.empty(int(n), dtype=torch.uint8, device=device)
            self._ws = {key: ws}          # keep one entry: batch sizes rarely alternate
        return ws

    def time_table(self, labels):
        """[n,5,1024] time-bias table for a vector of labels (= t*999), on the model's device."""
        h = self.handle()
        labels = labels.to(device=h.device, dtype=torch.float32).contiguous()
        table = torch.empty(labels.numel(), L.NUM_DENSE, L.HIDDEN, dtype=torch.float32, device=h.device)
        L.check(L.load().dpb_score_time_table(h.ptr, L.ptr(labels), labels.numel(), L.ptr(table),
                                              L.current_stream(h.device)))
        return table

    def raw_forward(self, x, labels, row_mult=None):
        """post_dense(...)(x) * row_mult.

        ``labels`` ([B] or [1], = t*999) and ``row_mult`` (None | [B] | [1]) are small schedule vectors: they
        are brought to the HOST once (a [B]-float copy) so that (a) the batch-uniform case is detected without
        a device reduction and (b) every schedule scalar is the CPU-fp32 value the reference would compute
        (``1 - exp(2 lmc)`` loses ~5e-4 relative at t=1e-3 to a single ulp of exp, so the device's exp must
        not be used for it).  The time path is evaluated once per distinct label."""
        self.check_width(x, 'batch')
        h = self.handle()
        L.require_cuda(x, 'batch')
        x = x.detach().to(torch.float32).contiguous()
        B = x.shape[0]
        out = torch.empty(B, self.pose_width, dtype=torch.float32, device=x.device)
        if B == 0:
            return out
        labels = labels.detach().to(device='cpu', dtype=torch.float32).reshape(-1)
        mult = None if row_mult is None else row_mult.detach().to(device='cpu', dtype=torch.float32).reshape(-1)
        uniform = labels.numel() == 1 or bool((labels == labels[0]).all())
        scale, rs, idx = 1.0, None, None
        if uniform:
            table = self.time_table(labels[:1])
            if mult is not None:
                if mult.numel() == 1 or bool((mult == mult[0]).all()):
                    scale = float(mult[0])
                else:
                    rs = mult.to(x.device)
        else:
            uniq, inv = torch.unique(labels, return_inverse=True)
            table, idx = self.time_table(uniq), inv.to(device=x.device, dtype=torch.int32).contiguous()
            rs = None if mult is None else mult.expand(B).contiguous().to(x.device)
        ws = self.workspace(B, x.device)
        L.check(L.load().dpb_score_forward(h.ptr, L.ptr(x), L.ptr(table), L.ptr(idx), L.ptr(rs), scale, L.ptr(out),
                                           B, self.engine, L.ptr(ws), ws.numel(), L.current_stream(x.device)))
        return out

    def check_width(self, x, name, rows=None):
        """``x`` must be [B, D] with D the network's pose width (63 axis-angle, 126 rot6d) and, if given, B = ``rows``:
        the kernels index every such buffer as [B, D], so a tensor of the other width must be rejected before them."""
        if x.dim() != 2 or x.shape[1] != self.pose_width or (rows is not None and x.shape[0] != rows):
            want = f'[{"B" if rows is None else rows}, {self.pose_width}]'
            raise ValueError(f'{name}: expected {want} for this {self.pose_width}-D score network, got {list(x.shape)}')

    @property
    def is_rot6d(self):
        return self.pose_width == L.POSE_DIM_ROT6D

    def forward(self, batch, t, condition=None, mask=None):
        """batch [B,D], t [B] (labels, i.e. t*999 when called through score_fn) -> [B,D]  (model.py:141-196);
        D = 63 (axis-angle) or 126 (rot6d)."""
        if self.training:
            raise NotImplementedError('ScoreModelFC.forward is the inference path; training goes through dposer_b200.losses '
                                      '(get_step_fn / get_sde_loss_fn: loss and gradients in one native call)')
        t = t.detach().to('cpu', torch.float32)
        row_mult = None
        if self.config.model.scale_by_sigma:
            used_sigmas = self._sigmas_host()[t.long()]    # model.py:159 (int64 gather, bit-exact)
            row_mult = 1.0 / used_sigmas
        return self.raw_forward(batch, t, row_mult)

    def _sigmas_host(self):
        if getattr(self, '_sig_cpu', None) is None or self._sig_cpu[1] != self.sigmas._version:
            self._sig_cpu = (self.sigmas.detach().cpu(), self.sigmas._version)
        return self._sig_cpu[0]
