"""Time the self-intersection metric (dposer_b200.metric.self_intersections_percentage) on the GPU: 500 meshes
(config 1's batch) and 65 536 SMPL-size meshes (UV spheres with seeded dents, 6890 vertices, 13 776 faces), CUDA
events after warm-up, next to the card's name and power limit and the float64 oracle's CPU time per mesh.
When pymeshlab happens to be importable, also compares its per-face selection with the kernel's on a few deformed
spheres (informational: parity with pymeshlab is not pinned).

    python scripts/si_time.py [--reps 5] [--out results/si_time.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dposer_b200 import metric, synthetic  # noqa: E402
from oracle import selfisect_ref as R  # noqa: E402


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f'nvidia-smi unavailable ({e})'
    return q


def time_batch(topo, v, reps):
    ws = torch.empty(topo.workspace_bytes(v.shape[0]), dtype=torch.uint8, device='cuda')
    for _ in range(2):
        topo.counts(v, None, ws)
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        cnt = topo.counts(v, None, ws)
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return ms, cnt


def pymeshlab_compare(vs, f):
    try:
        import pymeshlab
    except ImportError:
        return 'pymeshlab not importable: comparison skipped'
    sel = metric.self_intersections_percentage(torch.tensor(vs).cuda(), f, return_selection=True)[1].cpu().numpy()
    rows = []
    for r, v in enumerate(vs):
        try:
            ms = pymeshlab.MeshSet()
            ms.add_mesh(pymeshlab.Mesh(v.astype(np.float64), f.astype(np.int32)))
            ms.compute_selection_by_self_intersections_per_face()
            ref = ms.current_mesh().face_selection_array().astype(bool)
        except Exception as e:  # noqa: BLE001  (the filter's name differs across pymeshlab versions)
            return f'pymeshlab failed: {e}'
        rows.append(dict(row=r, kernel=int(sel[r].sum()), pymeshlab=int(ref.sum()), differ=int((sel[r] != ref).sum())))
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'si_time.py measures on the GPU'
    res = {'card (name, power limit, max SM clock)': card(), 'device': torch.cuda.get_device_name(0)}
    _, f = synthetic.uv_sphere()
    g = np.random.default_rng(0)
    n_geo = 64
    geo_np = np.stack([synthetic.dented_sphere(d, 1000 + r) for r, d in enumerate(g.uniform(0.9, 1.2, n_geo))])
    t = time.perf_counter()
    ref = [R.selection(geo_np[r], f)[1] for r in range(4)]
    res['oracle_cpu_s_per_mesh'] = (time.perf_counter() - t) / 4
    geo = torch.tensor(geo_np).cuda()
    topo = metric.MeshTopology(f, geo.shape[1])
    for B in (500, 65536):
        v = geo[torch.arange(B, device='cuda') % n_geo].contiguous()
        ms, cnt = time_batch(topo, v, args.reps)
        c = cnt[:4].cpu().numpy() * 100.0 / len(f)
        assert np.allclose(c, ref), (c, ref)
        res[f'B={B}'] = dict(ms=[round(x, 3) for x in ms], ms_median=float(np.median(ms)),
                             meshes_per_s=B / (np.median(ms) / 1e3), mean_si=float(cnt.double().mean() * 100 / len(f)))
        del v
    res['pymeshlab'] = pymeshlab_compare(geo_np[:4], f)
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or '.', exist_ok=True)
        with open(args.out, 'w') as fh:
            json.dump(res, fh, indent=1)


if __name__ == '__main__':
    main()
