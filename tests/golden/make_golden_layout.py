"""Mint tests/golden/layout.npz (room-layout post-processing) by running the REAL reference's inference() on CPU.

Run in the build container only (the GPU box has no /root/reference):
    python tests/golden/make_golden_layout.py
Writes only tests/golden/layout.npz (kept under 1 MB).  Shims: torchvision.resnet50 is forced to weights=None (no
network, as in make_golden.py), scipy.ndimage.filters / sklearn.decomposition are provided when missing, and shapely
(not installed) is replaced by the exact simple-ring predicate of oracle/layout_ref.py -- validity is therefore not
pinned to GEOS by this corpus.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = '/root/reference'
sys.path.insert(0, REF)

import torchvision.models as tvm            # noqa: E402
_orig = tvm.resnet50
tvm.resnet50 = lambda *a, **k: _orig(weights=None)     # no network (inference.py imports model.py)

# the 12-point example label of README_PREPARE_DATASET.md:53-64 (x, y): ceiling/floor pairs
CORNERS = np.array([[158, 186], [158, 329], [353, 185], [353, 330], [594, 154], [594, 363],
                    [713, 100], [713, 415], [692, 77], [692, 438], [965, 150], [965, 367]], np.float32)


def _layout_signals(cor, rs, bon_noise, cor_noise):
    """Boundary / corner signals of one labelled layout as the training targets define them (dataset.py:107-120,
    cor_2_1d :137-159; every corner counts as visible), with seeded noise and a random roll."""
    import dataset as ref_ds                                          # reference dataset.py
    H, W = 512, 1024
    bon = ref_ds.cor_2_1d(cor, H, W)
    corx = cor[:, 0]
    cols = np.arange(W)
    dist = np.min([np.abs(corx[:, None] - cols[None]), np.abs(corx[:, None] - cols[None] - W),
                   np.abs(corx[:, None] - cols[None] + W)], 0).min(0)
    y_cor = 0.96 ** dist
    bon = bon + rs.normal(0, bon_noise, bon.shape)
    y_cor = np.clip(0.9 * y_cor + rs.normal(0, cor_noise, y_cor.shape), 1e-4, 1 - 1e-4)   # few saturated ties
    shift = int(rs.randint(W))
    bon, y_cor = np.roll(bon, shift, -1), np.roll(y_cor, shift, -1)
    return bon.astype(np.float32), np.log(y_cor / (1 - y_cor)).astype(np.float32)


def golden_layout():
    """Room-layout post-processing (inference.py:95-139 with post_proc.py) minted by the real ``inference()`` on
    corner sets of the reference's own assets.  ``net`` is a stand-in returning prepared signals; what inference()
    hands to the post-processing (the decoded rows and sigmoid(cor)), the peaks, the walls, z1, cor_id, the fallback
    message and any exception are recorded.  shapely is not installed: Polygon.is_valid is the oracle's exact
    simple-ring predicate, so validity is not pinned to GEOS here."""
    import contextlib
    import glob
    import io
    import json
    import types
    from oracle import layout_ref
    for name in ('shapely', 'shapely.geometry'):
        sys.modules.setdefault(name, types.ModuleType(name))

    class _Polygon:
        def __init__(self, pts):
            self.is_valid = layout_ref.ring_is_valid(np.asarray(pts))
    sys.modules['shapely.geometry'].Polygon = _Polygon
    sys.modules['shapely.geometry'].LineString = object
    try:
        import scipy.ndimage.filters                                  # noqa: F401
    except Exception:
        import scipy.ndimage
        m = types.ModuleType('scipy.ndimage.filters')
        m.maximum_filter = scipy.ndimage.maximum_filter
        sys.modules['scipy.ndimage.filters'] = m
    try:
        import sklearn.decomposition                                  # noqa: F401  (post_proc imports PCA)
    except Exception:
        for name in ('sklearn', 'sklearn.decomposition'):
            sys.modules.setdefault(name, types.ModuleType(name))
        sys.modules['sklearn.decomposition'].PCA = object
    import inference as ref_inf
    from misc import post_proc as ref_pp

    rec = {}
    _peaks, _gen_ww, _fix_z = ref_inf.find_N_peaks, ref_pp.gen_ww, ref_pp.np_refine_by_fix_z

    def find_peaks(signal, **kw):
        rec['y_cor'] = signal.copy()
        out = _peaks(signal, **kw)
        rec['peaks'] = out[0].copy()
        return out

    def gen_ww(*a, **kw):
        cor, xy_cor = _gen_ww(*a, **kw)
        rec['types'] = np.array([c['type'] for c in xy_cor])
        rec['vals'] = np.array([c['val'] for c in xy_cor], np.float64)
        return cor, xy_cor

    def fix_z(c0, c1, z0):
        rec['y_bon'] = np.stack([c0, c1]).copy()
        res = _fix_z(c0, c1, z0)
        rec['z1'] = res[1]
        return res
    ref_inf.find_N_peaks, ref_pp.gen_ww, ref_pp.np_refine_by_fix_z = find_peaks, gen_ww, fix_z

    sets = []
    for path in sorted(glob.glob(os.path.join(REF, 'assets', 'inferenced', '*.json'))):
        uv = np.array(json.load(open(path))['uv'], np.float64)
        sets.append((os.path.basename(path)[:-5], uv * np.array([1024, 512])))
    sets.append(('readme_label', CORNERS.astype(np.float64)))
    rs = np.random.RandomState(2024)
    signals = []
    for name, cor in sets:
        signals.append((name, ) + _layout_signals(cor, rs, 0.004, 0.03))
    for k in range(12):                                               # harder: noisy rows, many spurious peaks
        name, cor = sets[k * 4]
        signals.append((name + '_hard', ) + _layout_signals(cor, rs, 0.03, 0.25))
    modes = [dict(), dict(force_cuboid=True)]
    extra = [dict(r=0.03), dict(min_v=0.3), dict(force_raw=True), dict(force_cuboid=True, min_v=0.97),
             dict(force_cuboid=True, r=0.07)]
    out = {k: [] for k in ('sig', 'force_cuboid', 'force_raw', 'min_v', 'r', 'status', 'fallback', 'z1', 'n_peaks',
                           'peaks', 'n_walls', 'types', 'n_cor', 'cor_id')}
    y_bons, y_cors, names = [], [], []
    cover, dropped = {}, 0
    for si, (name, bon, logit) in enumerate(signals):
        kws = modes + [extra[si % len(extra)]]
        y_bons_i = None
        for kw in kws:
            def net(x):
                return torch.from_numpy(bon[None].copy()), torch.from_numpy(logit[None, None].copy())
            rec.clear()
            err, msg = 0, io.StringIO()
            with contextlib.redirect_stderr(msg):
                try:
                    cor_id, z0, z1, _ = ref_inf.inference(net, torch.zeros(1, 3, 512, 1024), 'cpu', **kw)
                except AssertionError:
                    err = layout_ref.STATUS_ASSERT
                except ValueError:
                    err = layout_ref.STATUS_RING
            if y_bons_i is None:
                y_bons_i = rec['y_bon']
                if 'y_cor' not in rec:                                # force_raw first would skip peak finding
                    raise RuntimeError('the first mode must find peaks')
                y_bons.append(rec['y_bon']); y_cors.append(rec['y_cor']); names.append(name)
            layout_kw = {k: v for k, v in kw.items()}
            if layout_ref.near_tie(y_bons[-1], y_cors[-1], **layout_kw):
                dropped += 1
                continue
            o = layout_ref.layout(y_bons[-1], y_cors[-1], **layout_kw)
            fallback = 'Fail to generate valid general layout' in msg.getvalue()
            assert o['status'] == err and o['fallback'] == fallback, (name, kw)
            out['sig'].append(len(y_bons) - 1)
            out['force_cuboid'].append(bool(kw.get('force_cuboid', False)))
            out['force_raw'].append(bool(kw.get('force_raw', False)))
            out['min_v'].append(np.nan if kw.get('min_v') is None else kw['min_v'])
            out['r'].append(kw.get('r', 0.05))
            out['status'].append(err)
            out['fallback'].append(fallback)
            peaks = rec.get('peaks', np.zeros(0, np.int64)) if not kw.get('force_raw') else np.zeros(0, np.int64)
            types_ = rec.get('types', np.zeros(0, np.int64)) if not (err or kw.get('force_raw')) else np.zeros(0, np.int64)
            if err:
                cor_id, z1 = np.zeros((0, 2), np.float32), rec.get('z1', o['z1'])
            out['z1'].append(np.float64(z1))
            out['n_peaks'].append(len(peaks)); out['peaks'].append(np.asarray(peaks, np.int32))
            out['n_walls'].append(len(types_)); out['types'].append(np.asarray(types_, np.int8))
            out['n_cor'].append(len(cor_id)); out['cor_id'].append(np.asarray(cor_id, np.float32))
            mode = 'raw' if kw.get('force_raw') else 'cuboid' if kw.get('force_cuboid') else 'general'
            keys = [mode, 'r_px=%d' % int(round(1024 * kw.get('r', 0.05) / 2))]
            keys += ['min_v'] if kw.get('min_v') is not None else []
            keys += ['fallback'] if fallback else []
            keys += ['AssertionError'] if err == layout_ref.STATUS_ASSERT else []
            keys += ['ValueError'] if err == layout_ref.STATUS_RING else []
            keys += sorted(o['events']) if mode == 'general' else []
            for k in keys:
                cover[k] = cover.get(k, 0) + 1
    res = dict(y_bon=np.stack(y_bons).astype(np.float32), y_cor=np.stack(y_cors).astype(np.float32),
               names=np.array(names))
    for k in ('sig', 'n_peaks', 'n_walls', 'n_cor', 'status'):
        res[k] = np.array(out[k], np.int32)
    for k in ('force_cuboid', 'force_raw', 'fallback'):
        res[k] = np.array(out[k], bool)
    res['min_v'] = np.array(out['min_v'], np.float64)
    res['r'] = np.array(out['r'], np.float64)
    res['z1'] = np.array(out['z1'], np.float64)
    res['peaks'] = np.concatenate(out['peaks']).astype(np.int32)      # ragged: offsets from the n_* arrays
    res['types'] = np.concatenate(out['types']).astype(np.int8)
    res['cor_id'] = np.concatenate(out['cor_id']).astype(np.float32)
    path = os.path.join(HERE, 'layout.npz')
    np.savez_compressed(path, **res)
    print('layout golden: %d signals, %d cases (%d near-ties dropped), %d bytes' %
          (len(y_bons), len(out['sig']), dropped, os.path.getsize(path)))
    print('coverage', json.dumps(cover, sort_keys=True))
    needed = ['cuboid', 'general', 'raw', 'fallback', 'requeue', 'forced_infer', 'forced_change', 'min_v',
              'AssertionError', 'r_px=26', 'r_px=15']
    missing = [k for k in needed if not cover.get(k)]
    if missing:
        raise RuntimeError('layout corpus misses ' + ', '.join(missing))



if __name__ == '__main__':
    golden_layout()
