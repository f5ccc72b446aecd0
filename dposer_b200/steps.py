"""Native building blocks of the fitting loops: thin, allocation-free calls into libdposer_b200 on caller-owned
buffers (no autograd, no framework op per step).  The task loops in ``fitting.py`` / ``prior.py`` chain them by hand
-- the graph of each reference loop is fixed (run/completion.py:178-203, run/motion_denoising.py:226-268,
run/smplify.py:208-260) -- so a whole Adam step is ~8 kernel launches and can be captured in one CUDA graph.
"""
import ctypes as C

import torch

from . import _lib as L
from . import utils as mutils


def _p(t, offset=0):
    """Device pointer of element ``offset`` of a float32 tensor."""
    return None if t is None else C.c_void_p(t.data_ptr() + 4 * offset)


class Adam:
    """torch.optim.Adam(lr, betas=(0.9, 0.999), eps=1e-8) on a strided [rows, cols] view of ``buf`` starting at column
    ``col0`` (row stride = buf.shape[1]); state lives on the device, the update is one kernel (``dpb_adam_step``)."""

    def __init__(self, buf, col0, cols, lr, betas=(0.9, 0.999), eps=1e-8):
        assert buf.dtype == torch.float32 and buf.is_contiguous() and buf.dim() == 2
        self.buf, self.col0, self.cols, self.ld = buf, col0, cols, buf.shape[1]
        self.lr, self.b1, self.b2, self.eps = float(lr), float(betas[0]), float(betas[1]), float(eps)
        self.m = torch.zeros(buf.shape[0] * cols, dtype=torch.float32, device=buf.device)
        self.v = torch.zeros_like(self.m)
        self.t = 0

    def reset(self):
        """Fresh optimiser state on the same buffers (a new batch of problems; captured graphs stay valid)."""
        self.m.zero_()
        self.v.zero_()
        self.t = 0

    def step(self, g1, off1, ld1, s1=1.0, g2=None, off2=0, ld2=0, s2=0.0, col_scale2=None, g3=None, off3=0, ld3=0,
             s3=0.0):
        self.t += 1
        dev = self.buf.device
        L.check(L.load().dpb_adam_step(_p(self.buf, self.col0), self.ld, L.ptr(self.m), L.ptr(self.v), _p(g1, off1), ld1,
                                       float(s1), _p(g2, off2), ld2, float(s2), L.ptr(col_scale2), _p(g3, off3), ld3,
                                       float(s3), self.buf.shape[0], self.cols, self.lr, self.b1, self.b2, self.eps,
                                       self.t, L.current_stream(dev)))


class PriorStep:
    """DPoser prior loss value + closed-form gradient at one schedule entry, on preallocated buffers."""

    def __init__(self, model, sde, continuous, rows, device):
        self.model, self.sde, self.continuous = model, sde, continuous
        self.loss = torch.empty(1, dtype=torch.float32, device=device)
        self.grad = torch.empty(rows, model.pose_width, dtype=torch.float32, device=device)
        self.ws = model.workspace(rows, device)
        self.tables, self.scalars = None, None

    def schedule(self, times):
        """Precompute the time-bias tables [n,5,1024] and the host scalars for a list of times (python floats)."""
        self.scalars = [mutils.prior_scalars(self.sde, self.model, t, self.continuous) for t in times]
        labels = torch.cat([s['label'] for s in self.scalars])
        self.tables = self.model.time_table(labels)

    def __call__(self, x0, k, weighted, divisor, z=None, seed=0, step=0):
        ps = self.scalars[k]
        dev = x0.device
        L.check(L.load().dpb_prior_loss(self.model.handle().ptr, L.ptr(x0), L.ptr(self.tables[k]), ps['alpha'],
                                        ps['std'], ps['inv_sigma_std'], int(bool(weighted)), float(divisor), L.ptr(z),
                                        C.c_uint64(seed), C.c_uint64(step), L.ptr(self.loss), L.ptr(self.grad), None,
                                        x0.shape[0], self.model.engine, L.ptr(self.ws), self.ws.numel(),
                                        L.current_stream(dev)))
        return self.grad


class PriorInput:
    """How the fitting chains feed the prior from the axis-angle body pose, fixed by the score network's width:

    * 63-D (axis-angle): x0 = (pose - mean_poses) / std_poses, and Adam scales the prior's gradient by 1 / std.
    * 126-D (rot6d): x0 = normalize(axis_angle_to_rot6d(pose)) under ``Posenormalizer.column_affine()``, and the prior's
      gradient returns to the axis-angle pose through the VJP of that map."""

    def __init__(self, model, normalizer, rows, device):
        self.rot6d = model.pose_width == L.POSE_DIM_ROT6D
        mean, std = normalizer.column_affine() if self.rot6d else (normalizer.mean_poses, normalizer.std_poses)
        self.mean, self.std = mean.to(device).float().contiguous(), std.to(device).float().contiguous()
        self.inv_std = None if self.rot6d else (1.0 / self.std).contiguous()
        # the prior's gradient w.r.t. the axis-angle body pose
        self.g_axis = torch.zeros(rows, 63, dtype=torch.float32, device=device) if self.rot6d else None
        self.x0 = torch.zeros(rows, model.pose_width, dtype=torch.float32, device=device)

    def __call__(self, full_pose):
        """The prior's input from the body pose full_pose[:, 3:66], in ``self.x0``."""
        if self.rot6d:
            axis_to_rot6d_cols(full_pose, 3, self.mean, self.std, self.x0)       # offline_normalize(from_axis=True)
        else:
            affine_cols(full_pose, 3, full_pose.shape[1], self.mean, self.std, self.x0)
        return self.x0

    def adam_grad(self, full_pose, g):
        """``(g2, col_scale2)`` of ``Adam.step`` on the body pose from g, the prior's gradient w.r.t. x0."""
        if not self.rot6d:
            return g, self.inv_std
        axis_to_rot6d_cols_vjp(full_pose, 3, self.std, g, self.g_axis)
        return self.g_axis, None


class LbsStep:
    """LBS forward + backward on preallocated buffers (the autograd-free twin of body_model._LbsFn)."""

    def __init__(self, core, rows, device, need_verts, const_tail=True):
        self.core, self.rows, self.dev, self.need_verts = core, rows, torch.device(device), need_verts
        self.h = core.handle(device)
        f = lambda *s: torch.empty(*s, dtype=torch.float32, device=device)   # noqa: E731
        self.verts = f(rows, core.V, 3) if need_verts else None
        self.joints = f(rows, core.n_out, 3)
        self.g_verts = f(rows, core.V, 3) if need_verts else None
        self.g_joints = f(rows, core.n_out, 3)
        self.g_pose = f(rows, core.J * 3)
        self.g_shape = f(rows, core.S)
        self.g_transl = f(rows, 3)
        n = L.load().dpb_lbs_workspace_bytes(self.h.ptr, rows, 0)
        self.ws = torch.empty(int(n), dtype=torch.uint8, device=device)
        ns = int(L.load().dpb_lbs_backward_scratch_bytes(self.h.ptr, rows)) if need_verts else \
            (int(L.load().dpb_lbs_backward_scratch_bytes_joints(self.h.ptr, rows)) if rows >= 64 else 0)
        self.scratch = torch.empty(ns, dtype=torch.uint8, device=device) if ns else None
        self.flags = core.engine | (L.LBS_CONST_TAIL if (const_tail and core.tail is not None) else 0)

    def forward(self, shape, full_pose, transl, no_save=False):
        L.check(L.load().dpb_lbs_forward(self.h.ptr, L.ptr(shape), L.ptr(full_pose), L.ptr(transl), L.ptr(self.verts),
                                         L.ptr(self.joints), self.rows, self.flags | (L.LBS_NO_SAVE if no_save else 0),
                                         L.ptr(self.ws), self.ws.numel(), L.current_stream(self.dev)))

    def backward(self, shape, full_pose, use_verts, want_transl=False):
        L.check(L.load().dpb_lbs_backward(self.h.ptr, L.ptr(shape), L.ptr(full_pose),
                                          L.ptr(self.g_verts) if use_verts else None, L.ptr(self.g_joints),
                                          L.ptr(self.g_pose), L.ptr(self.g_shape),
                                          L.ptr(self.g_transl) if want_transl else None, self.rows, self.flags,
                                          L.ptr(self.ws), self.ws.numel(), L.ptr(self.scratch),
                                          0 if self.scratch is None else self.scratch.numel(),
                                          L.current_stream(self.dev)))


def affine_cols(x, off, ld, mean, std, out, inverse=False, out_off=0, out_ld=None, cols=None, squash=0.0):
    """out[:, out_off:out_off+cols] = (x[:, off:off+cols] - mean) / std   (or the inverse map; see dpb_affine_cols)."""
    cols = out.shape[1] if cols is None else cols
    L.check(L.load().dpb_affine_cols(_p(x, off), ld, L.ptr(mean), L.ptr(std), _p(out, out_off),
                                     out.shape[1] if out_ld is None else out_ld, out.shape[0], cols, int(inverse),
                                     float(squash), L.current_stream(out.device)))


def _rot6d_operands(x, off, rows, nj, per_joint, cols):
    """Checks of the rot6d calls, all before any library call: ``x`` [rows, ld] holds ``per_joint`` * nj input columns
    (3: axis-angle, 6: rot6d) from ``off``; ``cols`` lists (name, tensor, width): a [rows, width] matrix, or for width
    None the 6 * nj per-column statistics.  Shapes first (ValueError), then devices (RuntimeError for a CPU tensor)."""
    what = 'axis-angle' if per_joint == 3 else 'rot6d'
    if x.dim() != 2 or nj < 1 or x.shape[0] != rows or off < 0 or off + per_joint * nj > x.shape[1]:
        raise ValueError(f'x: expected {rows} rows holding {per_joint * nj} {what} columns from column {off}, '
                         f'got {list(x.shape)}')
    for name, t, width in cols:
        if (t.numel() != 6 * nj) if width is None else (list(t.shape) != [rows, width]):
            raise ValueError(f'{name}: expected {[6 * nj] if width is None else [rows, width]}, got {list(t.shape)}')
    named = [('x', x)] + [c[:2] for c in cols]
    for name, t in named:
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError(f'{name}: expected a contiguous float32 tensor, got {t.dtype}')
    for name, t in named:
        L.require_cuda(t, name)
        if t.device != x.device:
            raise ValueError(f'{name}: on {t.device}, x on {x.device}')


def axis_to_rot6d_cols(x, off, mean, std, out):
    """out[r, 6j:6j+6] = (rot6d(x[r, off+3j : off+3j+3]) - mean[6j:6j+6]) / std[6j:6j+6] for the out.shape[1] / 6
    joints (dpb_axis_to_rot6d_cols): the input of a rot6d prior from the axis-angle pose inside ``x``."""
    nj = out.shape[-1] // 6
    if out.dim() != 2 or out.shape[1] != 6 * nj:
        raise ValueError(f'out: expected 6 columns per joint, got {list(out.shape)}')
    _rot6d_operands(x, off, out.shape[0], nj, 3, [('out', out, 6 * nj), ('mean', mean, None), ('std', std, None)])
    L.check(L.load().dpb_axis_to_rot6d_cols(_p(x, off), x.shape[1], L.ptr(mean), L.ptr(std), L.ptr(out), out.shape[1],
                                            x.shape[0], nj, L.current_stream(x.device)))


def axis_to_rot6d_cols_vjp(x, off, std, g, g_x):
    """g_x [rows, 3 n] = the cotangent of x[:, off:off+3n] given g [rows, 6 n], the cotangent of axis_to_rot6d_cols'
    output (dpb_axis_to_rot6d_cols_vjp)."""
    nj = g.shape[-1] // 6
    if g.dim() != 2 or g.shape[1] != 6 * nj:
        raise ValueError(f'g: expected 6 columns per joint, got {list(g.shape)}')
    _rot6d_operands(x, off, g.shape[0], nj, 3, [('g', g, 6 * nj), ('g_x', g_x, 3 * nj), ('std', std, None)])
    L.check(L.load().dpb_axis_to_rot6d_cols_vjp(_p(x, off), x.shape[1], L.ptr(std), L.ptr(g), g.shape[1], L.ptr(g_x),
                                                g_x.shape[1], x.shape[0], nj, L.current_stream(x.device)))


def rot6d_to_axis_cols(x, off, mean, std, out):
    """out[r, 3j:3j+3] = rot6d_to_axis_angle(x[r, off+6j : off+6j+6] * std[6j:6j+6] + mean[6j:6j+6]) for the
    out.shape[1] / 3 joints (dpb_rot6d_to_axis_cols): the body pose of a rot6d network's normalised output."""
    nj = out.shape[-1] // 3
    if out.dim() != 2 or out.shape[1] != 3 * nj:
        raise ValueError(f'out: expected 3 columns per joint, got {list(out.shape)}')
    _rot6d_operands(x, off, out.shape[0], nj, 6, [('out', out, 3 * nj), ('mean', mean, None), ('std', std, None)])
    L.check(L.load().dpb_rot6d_to_axis_cols(_p(x, off), x.shape[1], L.ptr(mean), L.ptr(std), L.ptr(out), out.shape[1],
                                            x.shape[0], nj, L.current_stream(x.device)))


def rot6d_to_axis_cols_vjp(x, off, mean, std, g, g_x):
    """g_x [rows, 6 n] = the cotangent of x[:, off:off+6n] given g [rows, 3 n], the cotangent of rot6d_to_axis_cols'
    output (dpb_rot6d_to_axis_cols_vjp)."""
    nj = g.shape[-1] // 3
    if g.dim() != 2 or g.shape[1] != 3 * nj:
        raise ValueError(f'g: expected 3 columns per joint, got {list(g.shape)}')
    _rot6d_operands(x, off, g.shape[0], nj, 6, [('g', g, 3 * nj), ('g_x', g_x, 6 * nj), ('mean', mean, None),
                                                ('std', std, None)])
    L.check(L.load().dpb_rot6d_to_axis_cols_vjp(_p(x, off), x.shape[1], L.ptr(mean), L.ptr(std), L.ptr(g), g.shape[1],
                                                L.ptr(g_x), g_x.shape[1], x.shape[0], nj, L.current_stream(x.device)))


def motion_loss(lbs, target, seq_len, n_data, w_temp, w_data, seq_terms=None):
    L.check(L.load().dpb_motion_loss(L.ptr(lbs.verts), L.ptr(lbs.joints), L.ptr(target), lbs.rows, seq_len, lbs.core.V,
                                     lbs.core.n_out, n_data, float(w_temp), float(w_data), L.ptr(lbs.g_verts),
                                     L.ptr(lbs.g_joints), L.ptr(seq_terms), L.current_stream(lbs.dev)))


class StepGraphs:
    """One CUDA graph per step index of a fixed schedule: captured the first time a step runs on these buffers,
    replayed for every later batch of independent problems (chunks of sequences / images) that reuses them."""

    def __init__(self, enabled):
        self.enabled, self.graphs = enabled, {}

    def run(self, key, fn):
        if not self.enabled:
            fn()
            return
        g = self.graphs.get(key)
        if g is None:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                fn()
            self.graphs[key] = g
        g.replay()
