"""Time the Procrustes-aligned error kernel (dpb_procrustes, dposer_b200.metric.reconstruction_error) on the GPU at the
sizes users run: 131 072 x 49 SMPLify joint sets (config 5), 15 360 x 10 475 SMPL-X vertex sets (motion denoising,
config 4) and 65 536 x 6 890 SMPL vertex sets.  Each size is timed with and without the aligned points written, with
CUDA events after warm-up.  Every input is larger than L2 except the joint sets (154 MB, about L2's size), so the
figures are DRAM figures.  The achieved rate counts the bytes the algorithm needs: 24 B per point read (S1 and S2,
fp32), plus 12 B per point written with the aligned points; it is printed next to the HBM copy bandwidth SURVEY.md
measured (6 551.7 GB/s) and the card's name and power limit.

    python scripts/pa_time.py [--reps 20] [--out results/pa_time.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dposer_b200 import _lib as L  # noqa: E402

HBM_COPY_GBS = 6551.7
SIZES = [('SMPLify joints', 131072, 49), ('SMPL-X vertices', 15360, 10475), ('SMPL vertices', 65536, 6890)]


def card():
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f'nvidia-smi unavailable ({e})'


def launch(S1, S2, err, aligned):
    B, n = S1.shape[:2]
    L.check(L.load().dpb_procrustes(L.ptr(S1), L.ptr(S2), B, n, None, 0, L.ptr(err), L.ptr(aligned), None,
                                    L.current_stream(S1.device)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'pa_time.py measures on the GPU'
    res = {'card (name, power limit, max SM clock)': card(), 'device': torch.cuda.get_device_name(0)}
    g = torch.Generator(device='cuda').manual_seed(0)
    for name, B, n in SIZES:
        S1 = 0.3 * torch.randn(B, n, 3, generator=g, device='cuda')
        S2 = 1.1 * S1.flip(2) + 0.01 * torch.randn(B, n, 3, generator=g, device='cuda')
        err = torch.empty(B, device='cuda')
        for with_aligned in (False, True):
            aligned = torch.empty_like(S1) if with_aligned else None
            for _ in range(3):
                launch(S1, S2, err, aligned)
            torch.cuda.synchronize()
            ms = []
            for _ in range(args.reps):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                launch(S1, S2, err, aligned)
                b.record()
                b.synchronize()
                ms.append(a.elapsed_time(b))
            med = float(np.median(ms))
            gbs = B * n * (36 if with_aligned else 24) / (med * 1e-3) / 1e9
            res[f'{name} {B} x {n}' + (' + aligned' if with_aligned else '')] = dict(
                ms_median=round(med, 4), ms_min=round(min(ms), 4), ms_max=round(max(ms), 4), GB_per_s=round(gbs, 1),
                fraction_of_hbm_copy=round(gbs / HBM_COPY_GBS, 3))
            del aligned
        assert torch.isfinite(err).all()
        del S1, S2
        torch.cuda.empty_cache()
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or '.', exist_ok=True)
        with open(args.out, 'w') as fh:
            json.dump(res, fh, indent=1)


if __name__ == '__main__':
    main()
