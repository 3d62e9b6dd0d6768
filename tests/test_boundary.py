"""CPU: the drop-in boundary -- C ABI exports, checkpoint layout, loud failure without a GPU."""
import ctypes
import io
import os
import re
from collections import OrderedDict

import numpy as np
import pytest
import torch

import __graft_entry__ as entry
from horizonnet_b200 import _lib
from horizonnet_b200.model import HorizonNet
from horizonnet_b200.weights import synthetic_state_dict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def lib():
    entry.build()
    return _lib.lib()


def test_library_exports_every_symbol_of_the_header(lib):
    header = open(os.path.join(ROOT, 'include', 'horizonnet_b200.h')).read()
    declared = set(re.findall(r'\b(hn_[a-z0-9_]+)\s*\(', header))
    assert declared, 'no declarations found'
    for name in declared:
        assert hasattr(lib, name), f'{name} declared in include/horizonnet_b200.h but not exported'
    assert declared == set(_lib.SIGNATURES), 'ctypes signature table out of sync with the header'


def test_checkpoint_layout_round_trip():
    """reference misc/utils.py:49-65 save_model/load_trained_model, restated, on our class."""
    sd = synthetic_state_dict(3, 'random')
    net = HorizonNet('resnet50', True)
    net.load_state_dict(sd, strict=True)
    blob = io.BytesIO()
    torch.save(OrderedDict({'args': {}, 'kwargs': {'backbone': net.backbone, 'use_rnn': net.use_rnn},
                            'state_dict': net.state_dict()}), blob)
    blob.seek(0)
    ck = torch.load(blob, map_location='cpu')
    net2 = HorizonNet(**ck['kwargs'])
    net2.load_state_dict(ck['state_dict'])
    assert list(net2.state_dict().keys()) == list(sd.keys())
    for k, v in net2.state_dict().items():
        assert torch.equal(v, sd[k]), k


def test_checkpoint_round_trip_through_the_real_reference_utils(golden_dir, tmp_path):
    """The reference's OWN save_model / load_trained_model (misc/utils.py:49-65) applied to our class, unmodified, as
    recorded in tests/golden/checkpoint_ref_utils.json (make_golden.py golden_checkpoint): the same weights give the
    kwargs and the tensors (key, shape, dtype, sha256 of the bytes) save_model stored, and a checkpoint of the layout it
    wrote loads back into our class the way load_trained_model does it."""
    import hashlib
    import json

    def state_dict_digests(sd):                     # same record as make_golden.py state_dict_digests
        return [[k, list(v.shape), str(v.dtype), hashlib.sha256(v.detach().contiguous().numpy().tobytes()).hexdigest()]
                for k, v in sd.items()]
    g = json.load(open(os.path.join(golden_dir, 'checkpoint_ref_utils.json')))
    net = HorizonNet('resnet50', True)
    net.load_state_dict(synthetic_state_dict(g['weights_seed'], g['bn']), strict=True)
    assert {'backbone': net.backbone, 'use_rnn': net.use_rnn} == g['kwargs']          # utils.py:49-58 reads these
    assert state_dict_digests(net.state_dict()) == g['state_dict']
    assert g['loaded'] == {'class': 'HorizonNet', 'backbone': 'resnet50', 'use_rnn': True}
    path = str(tmp_path / 'ck.pth')
    parts = {'args': g['args'], 'kwargs': g['kwargs'], 'state_dict': net.state_dict()}
    torch.save(OrderedDict((k, parts[k]) for k in g['top_level']), path)
    ck = torch.load(path, map_location='cpu')
    net2 = HorizonNet(**ck['kwargs'])                                                  # utils.py:61-65 (strict load)
    net2.load_state_dict(ck['state_dict'])
    assert state_dict_digests(net2.state_dict()) == g['state_dict']


def test_train_mode_never_runs_the_eval_graph():
    """ADVICE round 1: net.train() (with or without torch.no_grad()) must not run the eval graph -- the reference uses
    batch statistics and dropout there (train.py:52).  forward() routes to the train-mode kernels (GPU only, so a CPU
    tensor is refused like in eval mode); the throughput / host entry points run the inference graph only and refuse."""
    net = HorizonNet('resnet50', True).train()
    assert net._train_mode_active()
    with torch.no_grad(), pytest.raises(RuntimeError, match='no CPU path'):
        net(torch.zeros(1, 3, 512, 1024))
    for call in (net.forward_pipelined, net.forward_host, net.submit_host):
        with pytest.raises(NotImplementedError):
            call(torch.zeros(1, 3, 512, 1024))
    # torch keeps the flag per module (train.py:251-256 mixes them): one BatchNorm2d in training mode is enough
    net.eval()
    assert not net._train_mode_active()
    net.feature_extractor.encoder.layer3[0].bn2.train()
    assert net._train_mode_active()
    net.eval().drop_out.train()
    assert net._train_mode_active()
    net.eval().bi_rnn.train()
    assert net._train_mode_active()


def test_module_surface_used_by_reference_callers():
    net = HorizonNet('resnet50', True)
    blocks = net.feature_extractor.list_blocks()            # train.py:202-208
    assert len(blocks) == 5 and len(blocks[0]) == 4
    assert sum(p.numel() for p in net.parameters()) == 81570348
    assert any(isinstance(m, torch.nn.BatchNorm2d) for m in net.modules())     # train.py:210-213
    assert any(isinstance(m, torch.nn.RNNBase) for m in net.modules())         # train.py:39-42
    assert net.linear.bias.tolist() == pytest.approx([-1] * 4 + [-0.478] * 4 + [0.425] * 4)
    with pytest.raises(NotImplementedError):
        HorizonNet('densenet169', True)                     # out of scope, fails loudly


def test_no_cpu_fallback():
    net = HorizonNet('resnet50', True).eval()
    with pytest.raises(NotImplementedError):
        net(torch.zeros(1, 3, 256, 512))                    # model.py:255-256
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            net(torch.zeros(1, 3, 512, 1024))
        from horizonnet_b200.misc.panostretch import pano_stretch
        with pytest.raises(RuntimeError):
            pano_stretch(np.zeros((8, 16, 3), np.float32), np.zeros((1, 2)), 1.0, 1.0)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, 'horizonnet_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh')):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle', src, re.M), f
                assert '/root/reference' not in src, f


def test_missing_device_is_reported_not_hidden(lib):
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    p = ctypes.c_void_p()
    assert lib.hn_model_create(0, 1, ctypes.byref(p)) != 0
    assert b'no CUDA device' in lib.hn_last_error()


def test_bench_reference_arm_prints_exactly_one_json_line():
    """bench.py contract: stdout carries ONE JSON line (the driver parses it); the reference arm runs on CPU.
    Everything else (progress, library banners) must go to stderr."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0', '--quick-cpu'],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'panoramas/sec' and d['unit'] == 'panoramas/s'
    assert d['value'] > 0 and d['higher_is_better'] is True
    assert d['cpu_baseline']['kind'] == 'port' and d['e2e']['h2d_bytes_per_step'] == 0
    # threads = CPUs this process may use, capped at physical cores and the cgroup quota (never os.cpu_count() blindly)
    ht = d['cpu_baseline']['host_threads']
    assert 1 <= d['cpu_baseline']['cores'] == ht['used'] <= ht['affinity']


def test_augmentation_draws_and_corner_bookkeeping_replay_the_reference(golden_dir):
    """Host logic of row f3 (no GPU): draw_params consumes np.random exactly like dataset.py:69-105 (the golden stores
    what the REAL dataset drew for these seeds) and augment_corners follows dataset.py:82, 91, 98."""
    from horizonnet_b200 import augment
    g = np.load(os.path.join(golden_dir, 'augment.npz'))
    for c, seed in enumerate((11, 12, 13, 14)):
        h, w = (int(v) for v in g[f'c{c}_hw'])
        pr = augment.draw_params(g[f'c{c}_cor_in'], w, rng=np.random.RandomState(seed))
        kx, ky, flip, dx, p = g[f'c{c}_params']
        assert (pr['kx'], pr['ky'], float(pr['flip']), float(pr['dx']), pr['p']) == (kx, ky, flip, dx, p)
        cor = augment.augment_corners(g[f'c{c}_cor_in'], h, w, pr['kx'], pr['ky'], pr['flip'], pr['dx'])
        assert np.abs(cor - g[f'c{c}_cor_out']).max() < 1e-3
    off = augment.draw_params(g['c0_cor_in'], 128, stretch=False, flip=False, rotate=False, gamma=False)
    assert off == dict(kx=None, ky=None, flip=False, dx=0, p=None)


def test_tracked_bench_line_carries_every_contract_key():
    """The last default `bench.py` line of the round (profiles/r02_bench_n1.json, copied from the GPU box) has every key
    the bench contract names, consistent with each other -- guards the JSON layout without needing a GPU."""
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    d = json.load(open(os.path.join(root, 'profiles', 'r02_bench_n1.json')))
    base = json.load(open(os.path.join(root, 'BASELINE.json')))
    for k in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline',
              'dtype', 'data', 'config', 'clocks', 'e2e', 'gpu_launches', 'roofline', 'cpu_baseline'):
        assert k in d, k
    assert base['metric'].startswith(d['metric']) and d['higher_is_better'] is True and d['scaling'] == 'weak' and d['data'] == 'synthetic'
    assert d['n_gpus'] == 1 and d['warmup'] >= 3 and d['gpu_launches'] > 0 and d['vs_baseline'] is None
    assert 'workload' in d['config'] and 'l2' in d['config'] and 'model' not in d['config']
    assert abs(d['value'] - d['config']['global_batch'] / d['ms_per_step'] * 1e3) < 1e-2 * d['value']
    for k in ('sm_mhz', 'sm_max_mhz', 'reasons'):
        assert k in d['clocks'], k
    assert not set(d['clocks']['reasons']) & {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'}
    e = d['e2e']
    assert e['unit'] == d['unit'] and e['h2d_bytes_per_step'] == 32 * 3 * 512 * 1024 * 4 and e['d2h_bytes_per_step'] == 32 * 3 * 1024 * 4
    assert e['value'] != d['value']                                   # measured separately, not a copy of the device-timed value
    r = d['roofline']
    for k in ('bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'):
        assert k in r, k
    assert r['bound'] in ('hbm', 'tensor') and abs(r['frac'] - r['achieved'] / r['peak']) < 1e-3
    c = d['cpu_baseline']
    for k in ('value', 'unit', 'cores', 'kind', 'sample'):
        assert k in c, k
    assert c['kind'] in ('reference', 'port') and c['unit'] == d['unit']
    t = d['aux']['train_step']
    assert t['wgrad_tc'] is True and abs(t['step_ms'] - (t['forward_ms'] + t['backward_ms'] + t['optimizer_ms'])) < 0.05


def test_every_environment_switch_of_the_library_is_documented():
    """Every HN_* variable the CUDA sources or the Python package read appears in INTEGRATION.md's switch table."""
    import glob
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    names = set()
    for f in glob.glob(os.path.join(root, 'horizonnet_b200', 'csrc', '*.cu*')) + glob.glob(os.path.join(root, 'horizonnet_b200', '*.py')):
        src = open(f).read()
        names |= set(re.findall(r'getenv\("(HN_[A-Z0-9_]+)"\)', src)) | set(re.findall(r"environ\.get\('(HN_[A-Z0-9_]+)'", src))
    doc = open(os.path.join(root, 'INTEGRATION.md')).read()
    assert len(names) >= 15
    missing = sorted(n for n in names if n not in doc)
    assert not missing, missing
