"""CPU: pin the oracle (oracle/) against golden outputs minted from the REAL reference
(tests/golden/make_golden.py).  Tolerances: forward 2e-5 max-abs on O(1) outputs (fp32 CPU
summation order differs between the functional restatement / machines; fp32-vs-fp64 noise floor
of the model is ~7e-7); pano_stretch 1.2e-7 (one fp32 ulp at values in [0,1))."""
import json
import os
import numpy as np
import pytest
import torch

from horizonnet_b200._spec import state_dict_spec
from horizonnet_b200.weights import synthetic_state_dict, synthetic_panoramas
from oracle import horizonnet_ref, panostretch_ref
from train_fixture import train_golden as _train_golden

KGRID = (0.5, 0.75, 1.0, 1.25, 1.5, 1.75, 2.0)


def test_spec_matches_reference_checkpoint_layout(golden_dir):
    ref = json.load(open(os.path.join(golden_dir, 'state_dict_keys.json')))
    spec = state_dict_spec()
    assert len(spec) == 448
    for (k, shape, dt), (k2, (s2, _)) in zip(ref, spec.items()):
        assert k == k2 and tuple(shape) == tuple(s2)
    n_params = sum(int(np.prod(s)) for k, (s, kind) in spec.items()
                   if kind not in ('bn_mean', 'bn_var', 'bn_count'))
    assert n_params == 81570348          # SURVEY 8b


def _sample(t, n=4096):
    flat = t.detach().reshape(-1).double().numpy()
    stride = max(1, flat.size // n)
    return flat[::stride][:n].astype(np.float32)


@pytest.mark.parametrize('name,bn', [('identity', 'identity'), ('randombn', 'random')])
def test_forward_oracle_matches_reference(golden_dir, name, bn):
    g = np.load(os.path.join(golden_dir, f'forward_{name}.npz'))
    sd = synthetic_state_dict(int(g['seed']), bn)
    x = synthetic_panoramas(int(g['batch']), seed=int(g['x_seed']))
    with torch.no_grad():
        bon, cor, stages = horizonnet_ref.forward(sd, x, return_stages=True)
    assert bon.shape == (x.shape[0], 2, 1024) and cor.shape == (x.shape[0], 1, 1024)
    assert np.abs(bon.numpy() - g['bon']).max() < 2e-5
    assert np.abs(cor.numpy() - g['cor']).max() < 2e-5
    for k, v in stages.items():
        ref = g[k + '_sample']
        scale = float(g[k + '_maxabs'])
        assert tuple(v.shape) == tuple(g[k + '_shape'])
        assert np.abs(_sample(v) - ref).max() <= 2e-6 * scale + 1e-6, k


def test_forward_oracle_rejects_other_sizes():
    sd = {}
    with pytest.raises(NotImplementedError):
        horizonnet_ref.forward(sd, torch.zeros(1, 3, 256, 512))


def test_panostretch_oracle_small_full_grid(golden_dir):
    g = dict(np.load(os.path.join(golden_dir, 'panostretch_small.npz')))
    g.update(np.load(os.path.join(golden_dir, 'panostretch_small_kx_above_1.npz')))
    img = g['img']
    for kx in KGRID:
        for ky in KGRID:
            out, _ = panostretch_ref.pano_stretch(img, np.zeros((1, 2), np.float32), kx, ky)
            assert out.dtype == np.float32 and out.shape == img.shape
            assert np.abs(out - g[f'out_{kx}_{ky}']).max() <= 1.2e-7, (kx, ky)
    out0, _ = panostretch_ref.pano_stretch(img, np.zeros((1, 2), np.float32), 1.5, 0.75, order=0)
    assert np.array_equal(out0, g['out0_1.5_0.75'])


def test_panostretch_oracle_full_size_rows_and_corners(golden_dir):
    g = np.load(os.path.join(golden_dir, 'panostretch_rows.npz'))
    img = np.random.RandomState(0).random_sample((512, 1024, 3)).astype(np.float32)
    corners = np.array([[158, 186], [158, 329], [353, 185], [353, 330], [594, 154], [594, 363],
                        [713, 100], [713, 415], [692, 77], [692, 438], [965, 150], [965, 367]], np.float32)
    rows = g['rows']
    for key in g.files:
        if not key.startswith('out_'):
            continue
        _, kx, ky = key.split('_')
        out, cor = panostretch_ref.pano_stretch(img, corners, float(kx), float(ky))
        assert np.abs(out[rows] - g[key]).max() <= 1.2e-7, key
        assert abs(out.astype(np.float64).sum() - float(g[f'sum_{kx}_{ky}'])) < 1e-3
        assert np.abs(cor - g[f'cor_{kx}_{ky}']).max() < 1e-9
    # identity property (SURVEY 8c): kx = ky = 1 reproduces the image
    out, cor = panostretch_ref.pano_stretch(img, corners, 1.0, 1.0)
    assert np.abs(out - img).max() <= 1.2e-7
    assert np.abs(cor - corners).max() < 1e-4


def test_legacy_wrap_rule():
    # SURVEY hard-part 5: scipy's legacy 'wrap' has period n-1: [10,20,30,40,50] at -0.3 -> 47.0
    a = np.array([[10., 20., 30., 40., 50.]])
    v = panostretch_ref.map_coordinates_wrap(a, np.array([[0.0]]), np.array([[-0.3]]))
    assert abs(float(v[0, 0]) - 47.0) < 1e-12


def test_tta_oracle_matches_reference(golden_dir):
    """oracle/tta_ref.py vs the reference's own augment / augment_undo / inference() (tests/golden/tta_randombn.npz)."""
    from oracle import tta_ref
    g = np.load(os.path.join(golden_dir, 'tta_randombn.npz'))
    sd = synthetic_state_dict(int(g['seed']), 'random')
    x = synthetic_panoramas(1, seed=int(g['x_seed']))
    y_bon, y_cor = tta_ref.tta_forward(sd, x, flip=bool(g['flip']), rotate=list(g['rotate']))
    assert np.abs(y_bon - g['y_bon']).max() < 5e-3          # pixel rows: 1e-5 rad * 512 / pi
    assert np.abs(y_cor - g['y_cor']).max() < 2e-5
    assert np.abs(g['cor_id'][0::2, 1] * 512 - y_bon[0]).max() < 5e-3


# ------------------------------------------------------------------------------- "next" rows f3 / f4
def _synthetic_u8(h, w, seed):
    return np.random.RandomState(seed).randint(0, 256, size=(h, w, 3)).astype(np.uint8)


def test_augment_oracle_matches_the_real_dataset_pipeline(golden_dir):
    """oracle/augment_ref.py against the tensor the REAL dataset.PanoCorBonDataset.__getitem__ produced
    (dataset.py:48-134, stretch + flip + rotate + gamma on).  1.2e-7 = one fp32 ulp below 1."""
    from oracle import augment_ref
    g = np.load(os.path.join(golden_dir, 'augment.npz'))
    for c in range(int(g['n_cases'])):
        h, w = (int(v) for v in g[f'c{c}_hw'])
        kx, ky, flip, dx, p = (float(v) for v in g[f'c{c}_params'])
        img = _synthetic_u8(h, w, int(g[f'c{c}_img_seed']))
        x = augment_ref.augment_image(img, kx, ky, bool(flip), int(dx), p)
        assert x.shape == (3, h, w) and x.dtype == np.float32
        got = x if h < 512 else x[:, g['rows']]
        assert np.abs(got - g[f'c{c}_x']).max() <= 1.2e-7, c
        assert abs(x.astype(np.float64).sum() - float(g[f'c{c}_sum'])) < 0.05, c
        cor = augment_ref.augment_corners(g[f'c{c}_cor_in'], h, w, kx, ky, bool(flip), int(dx))
        assert np.abs(cor - g[f'c{c}_cor_out']).max() < 1e-3, c          # float32 bookkeeping in the reference


def test_rotate_oracle_matches_the_real_rotatePanorama(golden_dir):
    from oracle import panorotate_ref
    g = np.load(os.path.join(golden_dir, 'rotate.npz'))
    out = panorotate_ref.rotate_panorama(g['small_img'], R=g['small_R'])
    assert out.dtype == np.float64 and np.abs(out - g['small_out']).max() < 1e-12
    out = panorotate_ref.rotate_panorama(g['small_img'], g['small_R'][2::-1])
    assert np.abs(out - g['small_out_vp']).max() < 1e-12
    img = np.random.RandomState(22).random_sample((512, 1024, 3)).astype(np.float32)
    for name in ('tilt', 'big'):
        o = panorotate_ref.rotate_panorama(img, R=g[f'{name}_R'])
        assert np.abs(o[g['rows']] - g[f'{name}_rows']).max() < 1e-12, name
        assert abs(o.sum() - float(g[f'{name}_sum'])) < 1e-6, name


# ------------------------------------------------------------------------------- train-mode forward (row f1, forward only)
@pytest.mark.parametrize('name', ['all', 'frozen1'])
def test_train_mode_oracle_matches_the_real_reference(golden_dir, name):
    """The oracle's TrainMode (batch-statistics BN + running update, both dropouts; frozen blocks like
    train.py:251-256, --bn_momentum like :210-213) against the REAL reference run under net.train(), with the masks
    the reference consumed."""
    g, sd, x, masks, running, frozen = _train_golden(golden_dir, name)
    tm = horizonnet_ref.TrainMode(masks=masks, momentum=float(g['momentum']), frozen=frozen)
    with torch.no_grad():
        bon, cor = horizonnet_ref.forward(sd, x, train=tm)
    assert np.abs(bon.numpy() - g['bon']).max() < 2e-5
    assert np.abs(cor.numpy() - g['cor']).max() < 2e-5
    assert len(frozen) == (0 if name == 'all' else 11)          # bn1 + layer1's 10 BatchNorm2d (blocks 0 and 1)
    for k, v in running.items():
        if k.rsplit('.', 1)[0] in frozen:
            assert torch.equal(v, sd[k]), k                      # the reference left frozen statistics alone
        else:
            assert torch.allclose(tm.running[k], v, rtol=1e-5, atol=1e-6), k
    assert set(tm.running) == {k for k in running if k.rsplit('.', 1)[0] not in frozen}
    assert g['num_batches_tracked'].sum() == 69 - len(frozen)


def test_train_mode_oracle_draws_the_reference_masks_from_torchs_generator(golden_dir):
    """masks=None: F.dropout in the reference's order reproduces, under the same torch.manual_seed, what the reference
    drew inside nn.LSTM and self.drop_out (CPU generator)."""
    g, sd, x, masks, _, _ = _train_golden(golden_dir, 'all')
    torch.manual_seed(int(g['train_seed']))
    with torch.no_grad():
        bon, cor = horizonnet_ref.forward(sd, x, train=horizonnet_ref.TrainMode())
    assert np.abs(bon.numpy() - g['bon']).max() < 2e-5 and np.abs(cor.numpy() - g['cor']).max() < 2e-5
    assert 0.49 < float((masks[0] > 0).float().mean()) < 0.51


@pytest.mark.parametrize('name,n_params,tol', [('backward', 241, 2e-4), ('backward_frozen1', 208, 1e-3)])
def test_oracle_backward_matches_the_real_reference(golden_dir, name, n_params, tol):
    """Row f1, backward: torch.autograd through the oracle's train-mode forward (the checker of the GPU whole-step tests)
    against the gradients the REAL reference's `loss.backward()` produced (train.py:53-56, :278; fixtures minted by
    tests/golden/make_golden.py golden_train_backward): loss and, for every parameter with a gradient, strided samples and
    |grad| max.  'backward_frozen1' = --freeze_earlier_blocks 1 (train.py:200-208, :251-256: 33 parameters frozen, their
    11 BatchNorm2d modules in eval mode).  Measured at mint time: 2.3e-5 / 2.1e-4 of the tensor max."""
    import torch.nn.functional as F
    from horizonnet_b200.weights import synthetic_state_dict, synthetic_panoramas
    g = np.load(os.path.join(golden_dir, f'train_{name}.npz'))
    batch, n = int(g['batch']), int(g['n'])
    sd = synthetic_state_dict(int(g['wseed']), 'random')
    x = synthetic_panoramas(batch, seed=int(g['x_seed']))
    gen = torch.Generator().manual_seed(int(g['y_seed']))
    y_bon, y_cor = torch.rand(batch, 2, 1024, generator=gen) - 0.5, torch.rand(batch, 1, 1024, generator=gen)
    torch.manual_seed(int(g['train_seed']))                  # the two dropout masks, in the reference's draw order
    masks = [torch.empty(256, batch, 1024).bernoulli_(0.5).div_(0.5) for _ in range(2)]
    names = [str(k) for k in g['names']]
    frozen = [str(k) for k in g['frozen']]
    assert len(names) == n_params and len(frozen) == (0 if n_params == 241 else 11)
    psd = {k: (v.clone().requires_grad_() if k in names else v) for k, v in sd.items()}
    bon, cor = horizonnet_ref.forward(psd, x, train=horizonnet_ref.TrainMode(masks=masks, frozen=frozen))
    loss = F.l1_loss(bon, y_bon) + F.binary_cross_entropy_with_logits(cor, y_cor)
    assert abs(loss.item() - float(g['loss'])) < 1e-6
    grads = torch.autograd.grad(loss, [psd[k] for k in names])
    gmax = float(g['absmax'].max())
    worst = 0.0
    for i, (k, gr) in enumerate(zip(names, grads)):
        flat = gr.reshape(-1)
        got = flat[::max(1, flat.numel() // n)][:n].numpy()
        scale = float(g['absmax'][i]) + 1e-4 * gmax          # conv biases in front of a train-mode BN: analytically zero gradient
        worst = max(worst, float(np.abs(got - g['samples'][i][:got.size]).max()) / scale,
                    abs(float(flat.abs().max()) - float(g['absmax'][i])) / scale)
    assert worst < tol, worst
