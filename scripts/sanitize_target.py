"""Small pass over every tcgen05 kernel and the LBS backward for `compute-sanitizer --tool memcheck` (run under gpurun)."""
import os, sys, torch
sys.path.insert(0, os.getcwd())
from dposer_b200 import _lib as L, sampling, sde_lib, synthetic
from dposer_b200.body_model import BodyModel
model = synthetic.make_score_model(42).cuda(); model.engine = L.ENGINE_TC
cfg = synthetic.default_config()
for B, N in [(300, 3), (19200, 2)]:
    fn = sampling.get_sampling_fn(cfg, sde_lib.subVPSDE(0.1, 20., N), (B, 63), lambda x: x, 1e-3, device='cuda')
    traj, x = fn(model, z=torch.randn(B, 63))
    torch.cuda.synchronize(); print('sampler ok', B, float(x.abs().mean()))
x = torch.randn(500, 63).cuda()
out = model(x, torch.full((500,), 300., device='cuda')); torch.cuda.synchronize(); print('fwd ok')
for mt, B in [('smpl', 200), ('smplx', 130)]:
    bm = BodyModel(synthetic.make_body_tensors(mt), batch_size=B, model_type=mt).cuda()
    inp = {k: v.cuda().requires_grad_(True) for k, v in synthetic.lbs_inputs(B, mt).items()}
    o = bm(**inp); (o.v.sum() + o.Jtr.sum()).backward(); torch.cuda.synchronize(); print('lbs ok', mt)
# round 2: joints-only tensor-core path (compact sub-model), score-net JVP, native fitting steps
for mt, B in [('smplx', 96), ('smpl', 130)]:
    bm = BodyModel(synthetic.make_body_tensors(mt), batch_size=B, model_type=mt).cuda()
    inp = {k: v.cuda().requires_grad_(True) for k, v in synthetic.lbs_inputs(B, mt).items()}
    o = bm(need_verts=False, **inp); o.Jtr.sum().backward(); torch.cuda.synchronize(); print('lbs joints-only ok', mt)
from dposer_b200 import likelihood
d, dv = likelihood.drift_and_div(model, sde_lib.subVPSDE(0.1, 20., 1000), torch.randn(70, 63).cuda(), 0.3,
                                 torch.randn(70, 63).cuda())
torch.cuda.synchronize(); print('jvp ok', float(dv.abs().mean()))
import types
from dposer_b200 import fitting
from dposer_b200.misc import Posenormalizer
mx = synthetic.make_body_tensors('smplx')
rows, L_ = 128, 8
bm = BodyModel(mx, num_betas=10, batch_size=rows, model_type='smplx').cuda()
norm = Posenormalizer(None, device='cuda', normalize=True, min_max=False, rot_rep='axis')
gt = synthetic.toy_poses()[:rows].cuda()
with torch.no_grad():
    jn = bm(pose_body=gt, need_verts=False).Jtr[:, :22]
md = fitting.MotionDenoise(cfg, types.SimpleNamespace(device='cuda'), model, bm, sde_lib.subVPSDE(0.1, 20., 1000), norm,
                           sde_N=500, batch_size=rows, seq_len=L_)
r = md.optimize(jn, time_strategy='3', sample_trun=4.0, iterations=1, steps_per_iter=2)
torch.cuda.synchronize(); print('motion denoise ok', bool(torch.isfinite(r['pose_body']).all()))
# round 2, training step (8(f) row 3): eager (side stream) and graph replay, ragged batch; the GEMM utility entry at ragged sizes
from dposer_b200 import losses
from dposer_b200.ema import ExponentialMovingAverage
cfg.optim.warmup = 2
tm = synthetic.make_score_model(42).cuda(); tm.train()
state = dict(optimizer=losses.get_optimizer(cfg, tm.parameters()), model=tm,
             ema=ExponentialMovingAverage(tm.parameters(), decay=cfg.model.ema_rate), step=0)
sde1k = sde_lib.subVPSDE(0.1, 20., 1000)
data = synthetic.toy_poses()[:200].cuda()
for graph in (False, True):
    fn = losses.get_step_fn(sde1k, True, losses.optimization_manager(cfg), reduce_mean=True, graph=graph)
    for i in range(3):
        ld = fn(state, data[:130 + 35 * (i % 2)])
    torch.cuda.synchronize(); print('train step ok graph=%s' % graph, float(ld['step_loss']))
import ctypes
lib = L.load()
for (M, N, K) in [(257, 129, 200), (63, 1024, 96)]:
    A, Bm, out = torch.randn(M, K).cuda(), torch.randn(N, K).cuda(), torch.empty(M, N).cuda()
    ws = torch.empty(int(lib.dpb_gemm_nt_workspace_bytes(M, N, K)), dtype=torch.uint8, device='cuda')
    L.check(lib.dpb_gemm_nt(L.ptr(A), L.ptr(Bm), None, L.ptr(out), M, N, K, L.ptr(ws), ws.numel(), L.current_stream(A.device)))
    torch.cuda.synchronize(); print('gemm ok', float((out - A @ Bm.T).abs().max()))
# device-side RK45 + tensor-core JVP: a short likelihood integration (loose tolerance) and the ODE sampler
from dposer_b200 import likelihood as lk
lfn = lk.get_likelihood_fn(sde1k, lambda v: v, rtol=1e-2, atol=1e-2, eps=1e-3)
model.eval()
bpd, zz, nfe = lfn(model, synthetic.toy_poses()[:70].cuda())
torch.cuda.synchronize(); print('likelihood rk45 ok', nfe, bool(torch.isfinite(bpd).all()))
ofn = sampling.get_ode_sampler(sde1k, (33, 63), lambda v: v, rtol=1e-2, atol=1e-2, eps=1e-3, device='cuda')
nfe, xo = ofn(model, z=torch.randn(33, 63))
torch.cuda.synchronize(); print('ode sampler rk45 ok', nfe, bool(torch.isfinite(xo).all()))
# auxiliary training loss: DDIM chain (forward / backward halves, gradient accumulation) + SMPL-X body terms
from dposer_b200.body_model import BodyModel as _BM2
from dposer_b200.misc import Posenormalizer
tm.train()
abm = _BM2(synthetic.make_body_tensors('smplx'), num_betas=10, batch_size=70, model_type='smplx').cuda()
anorm = Posenormalizer(None, device='cuda', normalize=True, min_max=False, rot_rep='axis')
afn = losses.get_step_fn(sde1k, True, losses.optimization_manager(cfg), reduce_mean=True, auxiliary_loss=True,
                         denormalize=anorm.offline_denormalize, body_model=abm, rot_rep='axis', denoise_steps=3)
for _ in range(2):
    ld = afn(state, anorm.offline_normalize(synthetic.toy_poses()[:70].cuda()))
torch.cuda.synchronize(); print('auxiliary step ok', float(ld['step_loss']), float(ld['v2v_loss']))
