"""Timing of the SMPL-X LBS forward (const tail: the CTA-pair fused kernel)."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from dposer_b200 import synthetic
from dposer_b200.body_model import BodyModel

B = int(os.environ.get('PROF_BL', 30720))
mt = os.environ.get('PROF_MODEL', 'smplx')
bm = BodyModel(synthetic.make_body_tensors(mt), batch_size=B, model_type=mt).cuda()
inp = {k: v.cuda() for k, v in synthetic.lbs_inputs(B, mt).items()}
flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
with torch.no_grad():
    for _ in range(3):
        bm(**inp)
    best = 1e9
    for _ in range(5):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); bm(**inp); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
print(f'{mt} B={B}: {best:.3f} ms  ({B/best*1e3/1e6:.2f} M poses/s)')
