"""Mint the golden fixtures by running the REAL reference (read-only, /root/reference) on CPU.

Run in the build container only (the GPU box has no /root/reference):
    python tests/golden/make_golden.py
Outputs (committed): tests/golden/forward_identity.npz, forward_randombn.npz,
panostretch_small.npz + panostretch_small_kx_above_1.npz, panostretch_rows.npz, tta_randombn.npz, augment.npz (row f3), rotate.npz (row f4),
train_all.npz / train_frozen1.npz (row f1, train-mode forward), train_backward.npz / train_backward_frozen1.npz (row f1, loss.backward()),
checkpoint_ref_utils.json (save_model / load_trained_model on our class).  The two shims are the ones SURVEY.md section 8c
describes: torchvision.resnet50 is forced to weights=None (no network), nothing else is patched.
Weights/inputs come from horizonnet_b200.weights (numpy RandomState => reproducible on any box).
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
tvm.resnet50 = lambda *a, **k: _orig(weights=None)     # shim 1: no network
import model as ref_model                    # noqa: E402  (reference model.py)
from misc import panostretch as ref_ps       # noqa: E402  (reference misc/panostretch.py)

from horizonnet_b200.weights import synthetic_state_dict, synthetic_panoramas   # noqa: E402

N_SAMPLES = 4096
KGRID = (0.5, 0.75, 1.0, 1.25, 1.5, 1.75, 2.0)
# the 12-point example label of README_PREPARE_DATASET.md:53-64 (x, y): ceiling/floor pairs
CORNERS = np.array([[158, 186], [158, 329], [353, 185], [353, 330], [594, 154], [594, 363],
                    [713, 100], [713, 415], [692, 77], [692, 438], [965, 150], [965, 367]], np.float32)


def sample(t):
    flat = t.detach().reshape(-1).double().numpy()
    stride = max(1, flat.size // N_SAMPLES)
    return flat[::stride][:N_SAMPLES].astype(np.float32), np.float64(np.abs(flat).mean()), np.float64(np.abs(flat).max())


def golden_forward(name, seed, bn, batch):
    torch.manual_seed(0)
    net = ref_model.HorizonNet('resnet50', True).eval()
    sd = synthetic_state_dict(seed, bn)
    net.load_state_dict(sd, strict=True)          # proves the 448-key layout is the reference's
    x = synthetic_panoramas(batch, seed=100 + seed)
    stages = {}
    net.feature_extractor.register_forward_hook(
        lambda m, i, o: stages.update({f'layer{j + 1}': o[j] for j in range(4)}))
    net.reduce_height_module.register_forward_hook(lambda m, i, o: stages.update(feature=o))
    net.bi_rnn.register_forward_hook(lambda m, i, o: stages.update(rnn_out=o[0]))
    with torch.no_grad():
        bon, cor = net(x)
    out = dict(bon=bon.numpy(), cor=cor.numpy(), seed=seed, batch=batch, x_seed=100 + seed)
    for k, v in stages.items():
        s, mean_abs, max_abs = sample(v)
        out[k + '_sample'] = s
        out[k + '_meanabs'] = mean_abs
        out[k + '_maxabs'] = max_abs
        out[k + '_shape'] = np.array(v.shape)
    np.savez_compressed(os.path.join(HERE, f'forward_{name}.npz'), **out)
    print(name, 'bon', float(bon.abs().max()), 'cor', float(cor.abs().max()),
          {k: float(v.abs().max()) for k, v in stages.items()})


def golden_panostretch():
    small = {}
    rs = np.random.RandomState(7)
    img_s = rs.random_sample((32, 64, 3)).astype(np.float32)
    small['img'] = img_s
    cs = CORNERS * np.array([64 / 1024, 32 / 512], np.float32)
    for kx in KGRID:
        for ky in KGRID:
            o, c = ref_ps.pano_stretch(img_s, cs, kx, ky)
            small[f'out_{kx}_{ky}'] = o
            small[f'cor_{kx}_{ky}'] = c
    o0, _ = ref_ps.pano_stretch(img_s, cs, 1.5, 0.75, order=0)
    small['out0_1.5_0.75'] = o0
    # two files of under 1 MB each: the kx > 1 half of the grid goes to the second
    upper = {k: small.pop(k) for k in list(small) if k.split('_')[0] in ('out', 'cor') and float(k.split('_')[1]) > 1.0}
    np.savez_compressed(os.path.join(HERE, 'panostretch_small.npz'), **small)
    np.savez_compressed(os.path.join(HERE, 'panostretch_small_kx_above_1.npz'), **upper)

    rows = {}
    img = np.random.RandomState(0).random_sample((512, 1024, 3)).astype(np.float32)
    sel = np.array([0, 1, 2, 130, 255, 256, 381, 509, 510, 511])
    rows['rows'] = sel
    for kx in KGRID:
        for ky in KGRID:
            o, c = ref_ps.pano_stretch(img, CORNERS, kx, ky)
            rows[f'sum_{kx}_{ky}'] = np.float64(o.astype(np.float64).sum())
            rows[f'sq_{kx}_{ky}'] = np.float64((o.astype(np.float64) ** 2).sum())
            rows[f'cor_{kx}_{ky}'] = c
            if (kx, ky) in ((2.0, 1.0), (0.5, 2.0), (1.0, 1.0), (1.25, 0.75), (2.0, 0.5), (0.75, 1.75)):
                rows[f'out_{kx}_{ky}'] = o[sel]
    np.savez_compressed(os.path.join(HERE, 'panostretch_rows.npz'), **rows)
    print('panostretch fixtures written')


def golden_tta():
    """TTA internals of reference inference.py:77-93, computed with the reference's own augment /
    augment_undo, plus the public inference(..., force_raw=True) result (its cor_id exposes y_bon_[0])."""
    import types
    for name in ('shapely', 'shapely.geometry'):                    # shim 2: not installed, never called with force_raw
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules['shapely.geometry'].Polygon = object
    sys.modules['shapely.geometry'].LineString = object
    try:
        import scipy.ndimage.filters                                 # noqa: F401  (removed in recent scipy)
    except Exception:
        import scipy.ndimage
        m = types.ModuleType('scipy.ndimage.filters')
        m.maximum_filter = scipy.ndimage.maximum_filter
        sys.modules['scipy.ndimage.filters'] = m
    import inference as ref_inf                                      # reference inference.py
    torch.manual_seed(0)
    net = ref_model.HorizonNet('resnet50', True).eval()
    net.load_state_dict(synthetic_state_dict(2, 'random'), strict=True)
    x = synthetic_panoramas(1, seed=102)
    flip, rotate = True, [0.25, 0.333]
    with torch.no_grad():
        xa, aug_type = ref_inf.augment(x, flip, rotate)
        y_bon_, y_cor_ = net(xa)
        y_bon_ = ref_inf.augment_undo(y_bon_.cpu(), aug_type).mean(0)
        y_cor_ = ref_inf.augment_undo(torch.sigmoid(y_cor_).cpu(), aug_type).mean(0)
        H = 512
        y_bon_ = (y_bon_[0] / np.pi + 0.5) * H - 0.5
        y_bon_[0] = np.clip(y_bon_[0], 1, H / 2 - 1)
        y_bon_[1] = np.clip(y_bon_[1], H / 2 + 1, H - 2)
        y_cor_ = y_cor_[0, 0]
        cor_id, z0, z1, _ = ref_inf.inference(net, x, 'cpu', flip=flip, rotate=rotate, force_raw=True)
    assert np.abs(cor_id[0::2, 1] * H - y_bon_[0]).max() < 1e-3      # the public function agrees with the restated lines
    np.savez_compressed(os.path.join(HERE, 'tta_randombn.npz'), y_bon=y_bon_.astype(np.float32),
                        y_cor=y_cor_.astype(np.float32), cor_id=cor_id, z1=np.float64(z1), seed=2, x_seed=102,
                        flip=flip, rotate=np.array(rotate))
    print('tta golden', y_bon_.min(), y_bon_.max(), float(y_cor_.max()))


def synthetic_u8(h, w, seed):
    """Smooth-ish synthetic uint8 RGB panorama (reproducible on any box)."""
    return np.random.RandomState(seed).randint(0, 256, size=(h, w, 3)).astype(np.uint8)


def golden_augment():
    """'next' row f3: the image tensor of the REAL dataset.PanoCorBonDataset.__getitem__ (dataset.py:48-134) with
    stretch + flip + rotate + gamma on, for a synthetic PNG and the README's 12-corner label.  np.random is seeded and
    the draws are replayed (same order as dataset.py:71-81, 88, 95, 102-104) to recover (kx, ky, flip, dx, p)."""
    import tempfile
    import types
    from PIL import Image
    for name in ('shapely', 'shapely.geometry'):
        sys.modules.setdefault(name, types.ModuleType(name))

    class _LineString:                               # occlusion labels only (dataset.py:182-195); not on the image path
        def __init__(self, pts): pass
        def intersects(self, other): return False
    sys.modules['shapely.geometry'].LineString = _LineString
    sys.modules['shapely.geometry'].Polygon = object
    import dataset as ref_ds                         # reference dataset.py
    _cdist = ref_ds.cdist                            # scipy >= 1.9 rejects p= for the default metric; label path only
    ref_ds.cdist = lambda a, b, p=1: _cdist(a, b, 'minkowski', p=p)
    out = {}
    sel = np.array([0, 1, 7, 100, 255, 256, 300, 411, 510, 511])
    out['rows'] = sel
    cases = []
    for case, (h, w, seed) in enumerate([(64, 128, 11), (512, 1024, 12), (512, 1024, 13), (512, 1024, 14)]):
        with tempfile.TemporaryDirectory() as root:
            os.makedirs(os.path.join(root, 'img')); os.makedirs(os.path.join(root, 'label_cor'))
            img = synthetic_u8(h, w, 500 + seed)
            Image.fromarray(img).save(os.path.join(root, 'img', 'pano.png'))
            cor = CORNERS * np.array([w / 1024, h / 512], np.float32)
            with open(os.path.join(root, 'label_cor', 'pano.txt'), 'w') as f:
                for x, y in cor:
                    f.write('%d %d\n' % (round(float(x)), round(float(y))))
            ds = ref_ds.PanoCorBonDataset(root, flip=True, rotate=True, gamma=True, stretch=True, return_cor=True)
            np.random.seed(seed)
            x, bon, y_cor, cor_out = ds[0]
            # replay the draws
            np.random.seed(seed)
            with open(os.path.join(root, 'label_cor', 'pano.txt')) as f:
                c0 = np.array([l.strip().split() for l in f if l.strip()], np.float32)
            c0 = np.roll(c0[:, :2], -2 * np.argmin(c0[::2, 0]), 0)
            xmin, ymin, xmax, ymax = ref_ds.cor2xybound(c0)
            kx = np.random.uniform(1.0, 2.0); ky = np.random.uniform(1.0, 2.0)
            kx = max(1 / kx, min(0.5 / xmin, 1.0)) if np.random.randint(2) == 0 else min(kx, max(10.0 / xmax, 1.0))
            ky = max(1 / ky, min(0.5 / ymin, 1.0)) if np.random.randint(2) == 0 else min(ky, max(10.0 / ymax, 1.0))
            flip = np.random.randint(2) == 0
            dx = np.random.randint(w)
            p = np.random.uniform(1, 2)
            if np.random.randint(2) == 0:
                p = 1 / p
        x = x.numpy()
        out[f'c{case}_hw'] = np.array([h, w]); out[f'c{case}_img_seed'] = 500 + seed
        out[f'c{case}_params'] = np.array([kx, ky, float(flip), float(dx), p], np.float64)
        out[f'c{case}_cor_in'] = c0; out[f'c{case}_cor_out'] = np.asarray(cor_out, np.float64)
        out[f'c{case}_sum'] = np.float64(x.astype(np.float64).sum()); out[f'c{case}_sq'] = np.float64((x.astype(np.float64) ** 2).sum())
        out[f'c{case}_x'] = x if h < 512 else x[:, sel]
        cases.append((h, w, kx, ky, flip, dx, p))
    out['n_cases'] = len(cases)
    np.savez_compressed(os.path.join(HERE, 'augment.npz'), **out)
    print('augment golden', cases)


def golden_rotate():
    """'next' row f4: the REAL misc/pano_lsd_align.rotatePanorama (only `pylsd` is stubbed: not installed, LSD line
    detection is not on this path)."""
    import types
    m = types.ModuleType('pylsd'); m.lsd = lambda *a, **k: None
    sys.modules.setdefault('pylsd', m)
    from misc import pano_lsd_align as ref_pl
    out = {}
    rs = np.random.RandomState(21)
    q, _ = np.linalg.qr(rs.randn(3, 3))
    small = rs.random_sample((32, 64, 3))
    out['small_img'] = small; out['small_R'] = q
    out['small_out'] = ref_pl.rotatePanorama(small, R=q)
    out['small_out_vp'] = ref_pl.rotatePanorama(small, q[2::-1])             # preprocess.py:65 call form
    img = np.random.RandomState(22).random_sample((512, 1024, 3)).astype(np.float32)
    sel = np.array([0, 1, 2, 77, 255, 256, 400, 509, 510, 511])
    out['rows'] = sel
    # a small tilt (the typical vanishing-point alignment) and a large rotation
    th = np.deg2rad(3.0)
    r_small = np.array([[np.cos(th), 0, np.sin(th)], [0, 1, 0], [-np.sin(th), 0, np.cos(th)]]) @ \
        np.array([[1, 0, 0], [0, np.cos(th / 2), -np.sin(th / 2)], [0, np.sin(th / 2), np.cos(th / 2)]])
    for name, R in (('tilt', r_small), ('big', q)):
        o = ref_pl.rotatePanorama(img, R=R)
        out[f'{name}_R'] = R; out[f'{name}_rows'] = o[sel]
        out[f'{name}_sum'] = np.float64(o.sum()); out[f'{name}_sq'] = np.float64((o ** 2).sum())
    np.savez_compressed(os.path.join(HERE, 'rotate.npz'), **out)
    print('rotate golden written')


TRAIN_SEED = 1234


def replay_dropout_masks(seed, batch, p=0.5):
    """The two masks the reference's train-mode forward consumes after torch.manual_seed(seed): at::dropout draws
    `empty_like(x).bernoulli_(1 - p).div_(1 - p)` -- first inside nn.LSTM on the layer-1 output [256, B, 1024]
    (model.py:226), then in self.drop_out on the LSTM output (model.py:265).  Nothing else on the path draws."""
    torch.manual_seed(seed)
    return [torch.empty(256, batch, 1024).bernoulli_(1 - p).div_(1 - p) for _ in range(2)]


def golden_train(name, freeze_earlier_blocks, bn_momentum=None, batch=2, wseed=1):
    """'next' row f1, forward only: the REAL reference under net.train() exactly as train.py drives it
    (:249 net.train(); :251-256 frozen blocks back to eval; :210-213 --bn_momentum), one forward (:52, without
    autocast: fp32 is the parity target).  Stores outputs, every BatchNorm2d's moved running statistics and the dropout
    masks (recovered by replaying torch's generator; the mint asserts that the oracle fed with those masks reproduces
    the reference to 2e-5 -- wrong masks would differ by O(1) -- which proves the replay)."""
    from oracle import horizonnet_ref as oracle
    net = ref_model.HorizonNet('resnet50', True)
    sd = synthetic_state_dict(wseed, 'random')
    net.load_state_dict(sd, strict=True)
    if bn_momentum:
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.momentum = bn_momentum                                # train.py:210-213
    net.train()                                                         # train.py:249
    frozen = []
    if freeze_earlier_blocks != -1:
        blocks = net.feature_extractor.list_blocks()
        for i in range(freeze_earlier_blocks + 1):
            for m in blocks[i]:
                m.eval()                                                # train.py:251-256
        frozen = [n for n, m in net.named_modules() if isinstance(m, torch.nn.BatchNorm2d) and not m.training]
    x = synthetic_panoramas(batch, seed=200 + wseed)
    torch.manual_seed(TRAIN_SEED)
    with torch.no_grad():
        bon, cor = net(x)
    after = net.state_dict()
    masks = replay_dropout_masks(TRAIN_SEED, batch)
    tm = oracle.TrainMode(masks=masks, momentum=bn_momentum or 0.1, frozen=frozen)
    with torch.no_grad():
        o_bon, o_cor = oracle.forward(sd, x, train=tm)
    err = max(float((o_bon - bon).abs().max()), float((o_cor - cor).abs().max()))
    assert err < 2e-5, f'mask replay / oracle restatement differs from the reference: {err}'   # wrong masks: O(1)
    bn_keys = [k for k in sd if k.endswith('running_mean') or k.endswith('running_var')]
    for k in bn_keys:
        moved = not torch.equal(after[k], sd[k])
        assert moved == (k.rsplit('.', 1)[0] not in frozen), k
        if moved:
            assert torch.allclose(tm.running[k], after[k], rtol=1e-5, atol=1e-6), k
    nbt = [int(after[k]) for k in after if k.endswith('num_batches_tracked')]
    out = dict(bon=bon.numpy(), cor=cor.numpy(), wseed=wseed, x_seed=200 + wseed, batch=batch, train_seed=TRAIN_SEED,
               momentum=np.float64(bn_momentum or 0.1), frozen=np.array(frozen, dtype='U'),
               masks_bits=np.packbits(np.stack([(m > 0).numpy() for m in masks]).reshape(-1)),
               running=np.concatenate([after[k].numpy().reshape(-1) for k in bn_keys]).astype(np.float32),
               num_batches_tracked=np.array(nbt))
    np.savez_compressed(os.path.join(HERE, f'train_{name}.npz'), **out)
    print('train golden', name, 'oracle-vs-reference', err, 'frozen BN modules:', len(frozen), 'bon', float(bon.abs().max()), 'cor', float(cor.abs().max()))


def golden_train_backward(name='backward', freeze_earlier_blocks=-1, batch=2, wseed=1, n=256):
    """Row f1, backward: the REAL reference's `loss.backward()` exactly as train.py drives it (:249 net.train(); :52 forward;
    :53-56 loss = L1(bon) + BCE-with-logits(cor); :278 backward), in fp32 without autocast.  Stores the loss and, for each
    of the 241 parameters, |grad| max, |grad| mean and `n` strided samples; the mint asserts that torch.autograd through the
    oracle (same dropout masks) reproduces them, which pins the oracle's backward -- the thing the GPU whole-step test
    compares the device gradients with -- to the reference."""
    import torch.nn.functional as F
    from oracle import horizonnet_ref as oracle
    net = ref_model.HorizonNet('resnet50', True)
    sd = synthetic_state_dict(wseed, 'random')
    net.load_state_dict(sd, strict=True)
    net.train()
    frozen = []
    if freeze_earlier_blocks != -1:                                          # train.py:200-208 and :251-256
        blocks = net.feature_extractor.list_blocks()
        for i in range(freeze_earlier_blocks + 1):
            for m in blocks[i]:
                m.eval()
                for p in m.parameters():
                    p.requires_grad = False
        frozen = [nm for nm, m in net.named_modules() if isinstance(m, torch.nn.BatchNorm2d) and not m.training]
    x = synthetic_panoramas(batch, seed=200 + wseed)
    g = torch.Generator().manual_seed(77)
    y_bon, y_cor = torch.rand(batch, 2, 1024, generator=g) - 0.5, torch.rand(batch, 1, 1024, generator=g)
    torch.manual_seed(TRAIN_SEED)
    bon, cor = net(x)
    loss = F.l1_loss(bon, y_bon) + F.binary_cross_entropy_with_logits(cor, y_cor)
    loss.backward()
    names = [k for k, p in net.named_parameters() if p.requires_grad]
    grads = {k: p.grad for k, p in net.named_parameters() if p.requires_grad}
    assert len(names) == (241 if not frozen else 241 - 33) and all(v is not None for v in grads.values())
    assert all(p.grad is None for p in net.parameters() if not p.requires_grad)
    # the oracle's autograd with the masks the reference consumed
    masks = replay_dropout_masks(TRAIN_SEED, batch)
    psd = {k: (v.clone().requires_grad_() if k in grads else v) for k, v in sd.items()}
    o_bon, o_cor = oracle.forward(psd, x, train=oracle.TrainMode(masks=masks, frozen=frozen))
    o_loss = F.l1_loss(o_bon, y_bon) + F.binary_cross_entropy_with_logits(o_cor, y_cor)
    o_grads = dict(zip(names, torch.autograd.grad(o_loss, [psd[k] for k in names])))
    gmax = max(float(v.abs().max()) for v in grads.values())
    worst = max(float((o_grads[k] - grads[k]).abs().max()) / (float(grads[k].abs().max()) + 1e-4 * gmax) for k in names)
    assert abs(loss.item() - o_loss.item()) < 1e-6 and worst < 1e-3, (loss.item(), o_loss.item(), worst)

    def strided(t):
        flat = t.detach().reshape(-1)
        stride = max(1, flat.numel() // n)
        out = np.zeros(n, np.float32)
        v = flat[::stride][:n].numpy()
        out[:v.size] = v
        return out
    np.savez_compressed(os.path.join(HERE, f'train_{name}.npz'), names=np.array(names, dtype='U'), loss=np.float64(loss.item()),
                        frozen=np.array(frozen, dtype='U'),
                        absmax=np.array([float(grads[k].abs().max()) for k in names]),
                        absmean=np.array([float(grads[k].abs().double().mean()) for k in names]),
                        samples=np.stack([strided(grads[k]) for k in names]), n=n, wseed=wseed, x_seed=200 + wseed, y_seed=77,
                        batch=batch, train_seed=TRAIN_SEED)
    print('train backward golden', name, ': loss', loss.item(), 'parameters with a gradient:', len(names), 'oracle autograd vs reference, worst tensor (rel. to its max):', worst)


def state_dict_digests(sd):
    """[key, shape, dtype, sha256 of the raw bytes] of every tensor, in the state_dict's order."""
    import hashlib
    return [[k, list(v.shape), str(v.dtype), hashlib.sha256(v.detach().contiguous().numpy().tobytes()).hexdigest()]
            for k, v in sd.items()]


def golden_checkpoint():
    """The REAL misc/utils.save_model / load_trained_model (utils.py:49-65) applied to our HorizonNet class, unmodified:
    the layout of the checkpoint save_model wrote (top-level keys, args, kwargs, a digest of every state_dict tensor)
    and what load_trained_model rebuilt from it."""
    import json
    import tempfile
    import types
    from misc import utils as ref_utils             # reference misc/utils.py
    from horizonnet_b200.model import HorizonNet
    net = HorizonNet('resnet50', True)
    net.load_state_dict(synthetic_state_dict(4, 'random'), strict=True)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, 'ck.pth')
        ref_utils.save_model(net, path, types.SimpleNamespace(lr=1e-4))          # args is vars()'d
        ck = torch.load(path, map_location='cpu')
        net2 = ref_utils.load_trained_model(HorizonNet, path)                      # strict load
    saved = state_dict_digests(ck['state_dict'])
    assert state_dict_digests(net2.state_dict()) == saved
    out = {'weights_seed': 4, 'bn': 'random', 'top_level': list(ck), 'args': ck['args'], 'kwargs': ck['kwargs'],
           'loaded': {'class': type(net2).__name__, 'backbone': net2.backbone, 'use_rnn': net2.use_rnn},
           'state_dict': saved}
    with open(os.path.join(HERE, 'checkpoint_ref_utils.json'), 'w') as f:         # one line per tensor
        head = json.dumps({k: v for k, v in out.items() if k != 'state_dict'})
        f.write(head[:-1] + ',\n"state_dict": [\n' + ',\n'.join(json.dumps(e) for e in saved) + '\n]}\n')
    print('checkpoint golden', out['top_level'], out['kwargs'], len(saved), 'tensors')


if __name__ == '__main__':
    if len(sys.argv) > 1 and sys.argv[1] == 'checkpoint':  # only the save_model / load_trained_model fixture
        golden_checkpoint()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == 'backward':    # only the backward fixtures of row f1
        golden_train_backward()
        golden_train_backward('backward_frozen1', 1)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == 'next':        # only the fixtures of the "next" rows f3 / f4
        golden_augment()
        golden_rotate()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == 'train':       # only the train-mode forward fixtures (row f1, forward)
        golden_train('all', -1)
        golden_train('frozen1', 1, bn_momentum=0.01)
        sys.exit(0)
    golden_augment()
    golden_rotate()
    golden_tta()
    golden_panostretch()
    golden_forward('identity', seed=0, bn='identity', batch=2)
    golden_forward('randombn', seed=1, bn='random', batch=1)
    golden_train('all', -1)
    golden_train('frozen1', 1, bn_momentum=0.01)
    golden_train_backward()
    golden_train_backward('backward_frozen1', 1)
    golden_checkpoint()
