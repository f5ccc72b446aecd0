"""Timing experiments on the fused LBS kernel: DPB_LBS_DEBUG masks in ONE process (run under `timeout`).
usage: python scripts/lbs_dbg.py "0 1 3 5 7 ..."
"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from dposer_b200 import synthetic
from dposer_b200.body_model import BodyModel
masks = [int(x) for x in (sys.argv[1] if len(sys.argv) > 1 else '0').split()]
B, mt = 65536, 'smpl'
bm = BodyModel(synthetic.make_body_tensors(mt), batch_size=B, model_type=mt).cuda()
inp = {k: v.cuda() for k, v in synthetic.lbs_inputs(B, mt).items()}
flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
with torch.no_grad():
    for m in masks:
        os.environ['DPB_LBS_DEBUG'] = str(m)
        for _ in range(2):
            bm(**inp)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(4):
            flush.fill_(1)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); bm(**inp); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        print(f'debug={m:3d}: {best:.3f} ms', flush=True)
