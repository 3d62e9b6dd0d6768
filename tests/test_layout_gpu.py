"""-m gpu: the device layout post-processing (hn_layout / hn_model_infer_layout) against the golden corpus minted from
the reference's inference(), against the oracle on seeded signals, for batch invariance, end to end through the
batched TTA forward, and through the CLI."""
import json
import os

import numpy as np
import pytest
import torch

import __graft_entry__ as entry
from horizonnet_b200 import _lib
from horizonnet_b200 import inference as hinf
from horizonnet_b200.model import HorizonNet
from horizonnet_b200.weights import synthetic_state_dict, synthetic_panoramas
from oracle import layout_ref
from test_layout import golden_cases

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.fixture(scope='module', autouse=True)
def _built():
    entry.build()
    _lib.lib()


def run_device(y_bon, y_cor, kw):
    """hn_layout on a batch of host signals -> list of per-panorama dicts (host numpy)."""
    yb = torch.from_numpy(np.ascontiguousarray(np.asarray(y_bon, np.float32).reshape(-1, 2, 1024))).to(DEV)
    yc = torch.from_numpy(np.ascontiguousarray(np.asarray(y_cor, np.float32).reshape(-1, 1024))).to(DEV)
    o = hinf.layout_device(yb, yc, **kw)
    torch.cuda.synchronize()
    st, nc = o['status'].cpu().numpy(), o['n_cor'].cpu().numpy()
    cor, z1 = o['cor_id'].cpu().numpy(), o['z1'].cpu().numpy()
    pk, tp = o['peaks'].cpu().numpy(), o['types'].cpu().numpy()
    return [dict(status=int(st[i, 0]), fallback=bool(st[i, 1]), peaks=pk[i, :st[i, 2]], types=tp[i, :st[i, 3]],
                 cor_id=cor[i, :nc[i]], z1=float(z1[i])) for i in range(len(nc))]


def assert_same(d, ref, what, cor_tol=1e-5):
    assert d['status'] == ref['status'] and d['fallback'] == ref['fallback'], what
    assert abs(d['z1'] - float(ref['z1'])) <= 1e-5 * abs(float(ref['z1'])), what
    if not ref.get('raw'):
        np.testing.assert_array_equal(d['peaks'], np.asarray(ref['peaks']), err_msg=what)
    if ref['status']:
        return
    if not ref.get('raw'):
        np.testing.assert_array_equal(d['types'], np.asarray(ref['types']), err_msg=what)
    assert d['cor_id'].shape == ref['cor_id'].shape, what
    assert np.abs(d['cor_id'] - ref['cor_id']).max() <= cor_tol, what


def test_golden_corpus(golden_dir):
    for i, c in enumerate(golden_cases(golden_dir)):
        d = run_device(c['y_bon'], c['y_cor'], c['kw'])[0]
        assert_same(d, dict(c, raw=c['kw']['force_raw']), 'golden case %d %s' % (i, c['kw']))


def seeded_signal(rs):
    """Boundary rows around a random room height with noise, and corner probabilities with 1-40 bumps, plateaus
    and noise."""
    W = 1024
    cols = np.arange(W)
    k = int(rs.randint(1, 41))
    ceil = 180 + 40 * np.sin(cols / W * 2 * np.pi * rs.randint(1, 6) + rs.uniform(0, 6)) + rs.normal(0, 2, W)
    floor = 330 - 40 * np.sin(cols / W * 2 * np.pi * rs.randint(1, 6) + rs.uniform(0, 6)) + rs.normal(0, 2, W)
    y_bon = np.stack([np.clip(ceil, 1, 255), np.clip(floor, 257, 510)]).astype(np.float32)
    centres = rs.choice(W, k, replace=False)
    d = np.min(np.abs(((cols[None] - centres[:, None]) + W // 2) % W - W // 2), 0)
    y_cor = 0.9 * 0.96 ** d + rs.uniform(0, 0.08, W)
    if rs.rand() < 0.3:                                          # plateaus: quantised values
        y_cor = np.round(y_cor * 20) / 20
    return y_bon, y_cor.astype(np.float32)


MODES = [dict(), dict(force_cuboid=True), dict(force_raw=True), dict(r=0.03), dict(min_v=0.3),
         dict(force_cuboid=True, r=0.07)]


def test_seeded_corpus_matches_oracle():
    rs = np.random.RandomState(123)
    checked = 0
    for n in range(400):
        y_bon, y_cor = seeded_signal(rs)
        kw = MODES[n % len(MODES)]
        if layout_ref.near_tie(y_bon, y_cor, vote_fn=layout_ref.vote_fast, **kw):
            continue
        ref = layout_ref.layout(y_bon, y_cor, vote_fn=layout_ref.vote_fast, **kw)
        d = run_device(y_bon, y_cor, kw)[0]
        assert_same(d, dict(ref, raw=kw.get('force_raw', False)), 'seeded %d %s' % (n, kw))
        checked += 1
    assert checked >= 256


def test_batch_invariance():
    rs = np.random.RandomState(7)
    sig = [seeded_signal(rs) for _ in range(32)]
    y_bon = np.stack([s[0] for s in sig])
    y_cor = np.stack([s[1] for s in sig])
    for kw in (dict(), dict(force_cuboid=True)):
        batch = run_device(y_bon, y_cor, kw)
        alone = run_device(y_bon[13], y_cor[13], kw)[0]
        for k in ('status', 'fallback', 'z1'):
            assert batch[13][k] == alone[k]
        for k in ('peaks', 'types', 'cor_id'):
            assert np.array_equal(batch[13][k], alone[k])


def _net():
    net = HorizonNet('resnet50', True).eval()
    net.load_state_dict(synthetic_state_dict(2, 'random'), strict=True)
    return net.to(DEV)


def test_infer_layout_end_to_end_bs32():
    net = _net()
    x = synthetic_panoramas(32, seed=300)
    flip, rotate = True, (0.25, 0.5)
    with torch.no_grad():
        out, y_bon, y_cor = hinf.infer_layout_device(net, x, flip=flip, rotate=rotate)
    torch.cuda.synchronize()
    y_bon, y_cor = y_bon.cpu().numpy(), y_cor.cpu().numpy()
    st, nc, cor = out['status'].cpu().numpy(), out['n_cor'].cpu().numpy(), out['cor_id'].cpu().numpy()
    z1 = out['z1'].cpu().numpy()
    for b in (0, 13, 31):                                        # the signals are tta_forward's, bit for bit
        tb, tc = hinf.tta_forward(net, x[b:b + 1], flip=flip, rotate=rotate)
        assert np.array_equal(tb, y_bon[b]) and np.array_equal(tc, y_cor[b]), b
    checked = 0
    for b in range(32):
        if layout_ref.near_tie(y_bon[b], y_cor[b], vote_fn=layout_ref.vote_fast):
            continue
        ref = layout_ref.layout(y_bon[b], y_cor[b], vote_fn=layout_ref.vote_fast)
        d = dict(status=int(st[b, 0]), fallback=bool(st[b, 1]), peaks=out['peaks'][b, :st[b, 2]].cpu().numpy(),
                 types=out['types'][b, :st[b, 3]].cpu().numpy(), cor_id=cor[b, :nc[b]], z1=float(z1[b]))
        assert_same(d, ref, 'panorama %d' % b)
        checked += 1
    assert checked >= 24


def test_cli_writes_the_same_json_as_inference(tmp_path):
    from PIL import Image
    net = _net()
    ckpt = tmp_path / 'net.pth'
    torch.save({'args': {}, 'kwargs': {'backbone': 'resnet50', 'use_rnn': True},
                'state_dict': synthetic_state_dict(2, 'random')}, str(ckpt))
    rs = np.random.RandomState(3)
    for name, (w, h) in (('a', (1024, 512)), ('b', (1024, 512)), ('c', (800, 400))):
        Image.fromarray(rs.randint(0, 256, (h, w, 3)).astype(np.uint8)).save(str(tmp_path / (name + '.png')))
    out_dir = tmp_path / 'out'
    hinf.main(['--pth', str(ckpt), '--img_glob', str(tmp_path / '*.png'), '--output_dir', str(out_dir),
               '--force_cuboid', '--flip', '--batch', '2'])
    for name in ('a', 'b', 'c'):
        x = hinf.load_image(str(tmp_path / (name + '.png')))
        with torch.no_grad():
            cor_id, z0, z1, _ = hinf.inference(net, x, DEV, flip=True, force_cuboid=True)
        got = json.load(open(os.path.join(str(out_dir), name + '.json')))
        assert got == {'z0': float(z0), 'z1': float(z1), 'uv': [[float(u), float(v)] for u, v in cor_id]}, name
