"""Layout post-processing benchmark (one GPU command):  python tools/layout_bench.py [--out profiles/r03_layout_bench.json]

Records, with the card's name and power limit:
  * hn_layout time per 32 panoramas (cuboid and general), CUDA events around each call, after warm-up, median of 300;
  * infer_layout end to end at batch 32 (no TTA, and flip + 2 rotations) against net(x) alone (same views);
  * the numpy oracle's per-panorama post-processing time on the same host (one thread).
Signals are the 32 first decoded signals of tests/golden/layout.npz (noisy layouts of real rooms)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import __graft_entry__ as entry                                        # noqa: E402
from horizonnet_b200 import inference as hinf                           # noqa: E402
from horizonnet_b200.model import HorizonNet                            # noqa: E402
from horizonnet_b200.weights import synthetic_state_dict, synthetic_panoramas   # noqa: E402
from oracle import layout_ref                                           # noqa: E402


def cuda_ms(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return float(np.median(out)), float(np.percentile(out, 10)), float(np.percentile(out, 90))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r03_layout_bench.json'))
    ap.add_argument('--iters', type=int, default=300)
    args = ap.parse_args()
    entry.build()
    assert torch.cuda.is_available(), 'layout_bench needs a GPU'
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {'gpu': smi[0] if smi else torch.cuda.get_device_name(0), 'batch': 32}

    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'layout.npz'))
    yb = torch.from_numpy(g['y_bon'][:32].copy()).cuda()
    yc = torch.from_numpy(g['y_cor'][:32].copy()).cuda()
    for name, kw in (('cuboid', dict(force_cuboid=True)), ('general', dict())):
        med, p10, p90 = cuda_ms(lambda: hinf.layout_device(yb, yc, **kw), 20, args.iters)
        res['hn_layout_ms_per_32_' + name] = {'median': med, 'p10': p10, 'p90': p90}

    net = HorizonNet('resnet50', True).eval()
    net.load_state_dict(synthetic_state_dict(0, 'random'), strict=True)
    net = net.to('cuda:0')
    x = synthetic_panoramas(32, seed=11).cuda()
    with torch.no_grad():
        for name, flip, rot in (('no_tta', False, ()), ('flip_rot2', True, (0.25, 0.5))):
            views = 1 + int(flip) + len(rot)
            # net(x) alone on the same 32 * views views, in forwards of 32 like infer_layout's chunks
            med_net = cuda_ms(lambda: [net(x) for _ in range(views)], 3, 20)[0]
            med_e2e = cuda_ms(lambda: hinf.infer_layout_device(net, x, flip=flip, rotate=rot, force_cuboid=True), 3, 20)[0]
            res['infer_layout_bs32_' + name] = {'infer_layout_ms': med_e2e, 'net_forward_same_views_ms': med_net,
                                                'views_per_panorama': views}

    cpu = {}
    for name, kw in (('cuboid', dict(force_cuboid=True)), ('general', dict())):
        t = []
        for i in range(32):
            t0 = time.perf_counter()
            layout_ref.layout(g['y_bon'][i], g['y_cor'][i], vote_fn=layout_ref.vote, **kw)
            t.append(time.perf_counter() - t0)
        cpu[name] = float(np.median(t) * 1e3)
    res['oracle_cpu_ms_per_panorama'] = cpu
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
