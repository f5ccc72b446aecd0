"""A/B of the L2 policy bits of lt3::lbs_fused3_kernel (DPB_LBS_DEBUG: 16 = WITHOUT L2::evict_last on the basis / weight
loads, 32 = WITHOUT st.global.cs vertex stores; the results do not change): bit-compare the vertices and time each variant.
usage: python scripts/lbs_hint_ab.py [B]      (each variant runs in a child with a timeout)"""
import os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# child process: time the forward and save a sample of the vertices
CHILD = r'''
import os, sys, torch
sys.path.insert(0, %r)
from dposer_b200 import synthetic
from dposer_b200.body_model import BodyModel
mt, B, out = sys.argv[1], int(sys.argv[2]), sys.argv[3]
bm = BodyModel(synthetic.make_body_tensors(mt), batch_size=B, model_type=mt).cuda()
inp = {k: v.cuda() for k, v in synthetic.lbs_inputs(B, mt).items()}
flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
with torch.no_grad():
    for _ in range(3):
        o = bm(**inp)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(5):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); o = bm(**inp); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    v = o.v
    idx = torch.arange(0, B, max(1, B // 997), device='cuda')
    torch.save({'ms': best, 'sum': float(v.double().sum()), 'abs': float(v.double().abs().sum()), 'rows': v[idx].cpu(),
                'nan': bool(torch.isnan(v).any())}, out)
print('ok', best)
''' % ROOT


def run(B, dbg, tag):
    out = f'/tmp/lbs_hint_{tag}.pt'
    env = dict(os.environ, DPB_LBS_DEBUG=str(dbg))
    try:
        r = subprocess.run([sys.executable, '-c', CHILD, 'smpl', str(B), out], env=env, timeout=60, capture_output=True, text=True)
    except subprocess.TimeoutExpired:
        return None, 'HANG (killed after 60 s)'
    if r.returncode != 0:
        return None, r.stderr[-600:]
    import torch
    return torch.load(out), ''


if __name__ == '__main__':
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
    base = None
    for rnd in range(2):
        for dbg in (0, 16, 32, 48):
            d, err = run(B, dbg, f'{dbg}_{rnd}')
            if d is None:
                print(f'debug={dbg}: {err}', flush=True)
                continue
            if base is None:
                base = d
            diff = float((d['rows'] - base['rows']).abs().max())
            print(f'round {rnd} debug={dbg}: {d["ms"]:.3f} ms  nan={d["nan"]}  max|diff vs debug=0|={diff}', flush=True)
