"""-m gpu: parity of the CUDA path (through the C ABI) against the CPU oracle, the committed
golden fixtures (minted from the real reference) and size-independent properties.

Tolerances: forward outputs 1e-4 max-abs (BASELINE north_star), kernel unit tests relative to the
output scale; pano_stretch 1.2e-7 (one fp32 ulp in [0,1): 'pixel-exact to bilinear rounding')."""
import os
import numpy as np
import pytest
import torch

import __graft_entry__ as entry
from horizonnet_b200 import _lib
from horizonnet_b200.model import HorizonNet
from horizonnet_b200.misc.panostretch import pano_stretch, pano_stretch_batch
from horizonnet_b200.weights import synthetic_state_dict, synthetic_panoramas
from oracle import horizonnet_ref, panostretch_ref
import gpu_utils as gu

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
KGRID = (0.5, 0.75, 1.0, 1.25, 1.5, 1.75, 2.0)


@pytest.fixture(scope='module', autouse=True)
def _built():
    entry.build()
    _lib.lib()


def _net(sd, tensor_cores):
    net = HorizonNet('resnet50', True).eval()
    net.load_state_dict(sd, strict=True)
    net.use_tensor_cores(tensor_cores)
    return net.to(DEV)


# ------------------------------------------------------------------------------- conv kernels
CONV_CASES = [
    # B, Cin, H, W, Cout, k, stride, bias/bn, residual, relu
    (2, 64, 8, 32, 64, 1, (1, 1), False, True),
    (1, 64, 16, 32, 256, 1, (1, 1), True, True),       # conv3 + identity + relu
    (2, 32, 9, 32, 48, 3, (1, 1), False, True),        # odd H, Cout not a multiple of 64
    (2, 128, 16, 64, 128, 3, (2, 2), False, True),     # stride-2 3x3 (layer2.0.conv2)
    (1, 256, 16, 32, 512, 1, (2, 2), False, False),    # stride-2 downsample
    (2, 64, 16, 32, 32, 3, (2, 1), False, True),       # GHC conv, stride (2,1)
    (3, 512, 2, 32, 256, 3, (2, 1), False, True),      # H 2 -> 1
    (1, 1024, 4, 32, 4096, 1, (1, 1), False, False),   # LSTM projection shape family
    (2, 512, 8, 32, 256, 3, (1, 1), False, True),      # large-K 3x3, conv mode, multi-row tiles
    (1, 512, 9, 62, 256, 1, (1, 1), True, True),       # K=512 1x1 with residual: GEMM mode of conv_tc_kernel, odd tile count
    (3, 256, 16, 64, 128, 3, (2, 1), False, True),     # stride (2,1), two rows per tile
    (1, 64, 5, 256, 64, 3, (1, 1), False, True),       # W >= 128: single-row tiles, dx taps share one 130-pixel input row
    (2, 128, 6, 128, 256, 3, (2, 1), True, True),      # same with stride (2,1) and bias (GHC on layer1/2 features)
]


@pytest.mark.parametrize('impl', [0, 1])
@pytest.mark.parametrize('case', CONV_CASES)
def test_conv_kernel_vs_torch(case, impl):
    B, Ci, H, W, Co, k, stride, residual, relu = case
    g = torch.Generator().manual_seed(hash(case) % (2 ** 31))
    x = torch.randn(B, Ci, H, W, generator=g)
    w = torch.randn(Co, Ci, k, k, generator=g) / (Ci * k * k) ** 0.5
    scale = torch.rand(Co, generator=g) + 0.5
    shift = torch.randn(Co, generator=g) * 0.1
    Ho = (H + 2 * (k // 2) - k) // stride[0] + 1
    Wo = (W + 2 * (k // 2) - k) // stride[1] + 1
    res = torch.randn(B, Co, Ho, Wo, generator=g) if residual else None
    ref = gu.conv2d_reference(x, w, scale, shift, stride, k // 2, k // 2, relu, res)
    try:
        y, raw = gu.conv2d(x.to(DEV), w.to(DEV), scale.to(DEV), shift.to(DEV), stride, k // 2, k // 2, relu,
                           res.to(DEV) if res is not None else None, impl=impl)
    except RuntimeError as e:
        if impl == 1 and 'not supported by the tcgen05 kernel' in str(e):
            pytest.skip('shape not covered by the tensor-core kernel (fp32 kernel covers it)')
        raise
    tol = 2e-5 if impl == 0 else 1e-4       # fp32 exact path / split-bf16 3-product path
    err = (y.cpu().double() - ref).abs().max().item()
    assert err <= tol * max(1.0, ref.abs().max().item()), err
    # halo columns must be the circular wrap of the interior
    assert torch.equal(raw[:, :, 0], raw[:, :, -2]) and torch.equal(raw[:, :, -1], raw[:, :, 1])


# ------------------------------------------------------------------------------- LSTM kernel
@pytest.mark.parametrize('T,B', [(5, 1), (24, 7), (16, 32), (12, 40)])
def test_lstm_layer_vs_oracle(T, B):
    g = torch.Generator().manual_seed(T * 100 + B)
    xproj = torch.randn(T, B, 4096, generator=g) * 0.5
    whh = [torch.rand(2048, 512, generator=g) * 0.08 - 0.04 for _ in range(2)]
    zero = torch.zeros(2048)
    ref = []
    for d in range(2):
        # oracle recurrence with the projection already applied: feed identity input weights
        xp = xproj[:, :, d * 2048:(d + 1) * 2048]
        h = torch.zeros(B, 512); c = torch.zeros(B, 512)
        out = torch.empty(T, B, 512)
        for t in (range(T - 1, -1, -1) if d else range(T)):
            gates = xp[t] + h @ whh[d].t()
            i, f, gg, o = gates.chunk(4, dim=1)
            c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
            h = torch.sigmoid(o) * torch.tanh(c)
            out[t] = h
        ref.append(out)
    ref = torch.cat(ref, dim=2)
    out = torch.full((T, B, 1024), float('nan'), device=DEV)
    xd, w0, w1 = xproj.to(DEV), whh[0].to(DEV), whh[1].to(DEV)
    rc = _lib.lib().hn_lstm_layer(xd.data_ptr(), w0.data_ptr(), w1.data_ptr(), out.data_ptr(), T, B,
                                  torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, 'hn_lstm_layer')
    torch.cuda.synchronize()
    assert (out.cpu() - ref).abs().max().item() < 2e-6


def test_lstm_layer_matches_oracle_function():
    """The oracle's own lstm_layer_dir (incl. input projection) against GEMM-free kernel input."""
    g = torch.Generator().manual_seed(11)
    T, B = 9, 3
    x = torch.randn(T, B, 64, generator=g)
    wih = [torch.randn(2048, 64, generator=g) * 0.1 for _ in range(2)]
    whh = [torch.randn(2048, 512, generator=g) * 0.04 for _ in range(2)]
    bih = [torch.randn(2048, generator=g) * 0.1 for _ in range(2)]
    bhh = [torch.randn(2048, generator=g) * 0.1 for _ in range(2)]
    ref = torch.cat([horizonnet_ref.lstm_layer_dir(x, wih[d], whh[d], bih[d], bhh[d], bool(d)) for d in range(2)], 2)
    xproj = torch.cat([x @ wih[d].t() + bih[d] + bhh[d] for d in range(2)], dim=2).to(DEV)
    out = torch.empty(T, B, 1024, device=DEV)
    w0, w1 = whh[0].to(DEV), whh[1].to(DEV)
    _lib.check(_lib.lib().hn_lstm_layer(xproj.data_ptr(), w0.data_ptr(), w1.data_ptr(), out.data_ptr(), T, B, None),
               'hn_lstm_layer')
    torch.cuda.synchronize()
    assert (out.cpu() - ref).abs().max().item() < 2e-6


# ------------------------------------------------------------------------------- forward
@pytest.mark.parametrize('tensor_cores', [False, True])
@pytest.mark.parametrize('name,bn', [('identity', 'identity'), ('randombn', 'random')])
def test_forward_matches_reference_golden(golden_dir, name, bn, tensor_cores):
    g = np.load(os.path.join(golden_dir, f'forward_{name}.npz'))
    sd = synthetic_state_dict(int(g['seed']), bn)
    net = _net(sd, tensor_cores)
    x = synthetic_panoramas(int(g['batch']), seed=int(g['x_seed']))
    with torch.no_grad():
        bon, cor = net(x.to(DEV))
    bon, cor = bon.cpu().numpy(), cor.cpu().numpy()
    net.check()
    # per-stage samples first: they localise a failure
    for stage in ('layer1', 'layer2', 'layer3', 'layer4', 'feature', 'rnn_out'):
        v = net.debug_stage(stage).cpu()
        assert tuple(v.shape) == tuple(g[stage + '_shape']), stage
        flat = v.reshape(-1).numpy()
        stride = max(1, flat.size // 4096)
        got = flat[::stride][:4096]
        scale = float(g[stage + '_maxabs'])
        tol = (2e-5 if not tensor_cores else 2e-4) * scale + 1e-6
        assert np.abs(got - g[stage + '_sample']).max() <= tol, stage
    assert np.abs(bon - g['bon']).max() < 1e-4
    assert np.abs(cor - g['cor']).max() < 1e-4


@pytest.mark.parametrize('tensor_cores', [False, True])
def test_forward_matches_oracle_and_is_batch_invariant(tensor_cores):
    sd = synthetic_state_dict(7, 'random')
    net = _net(sd, tensor_cores)
    x = synthetic_panoramas(3, seed=21, channels=4)          # extra channel must be ignored (model.py:252)
    with torch.no_grad():
        bon3, cor3 = net(x.to(DEV))
        bon1, cor1 = net(x[1:2].to(DEV))
        rbon, rcor = horizonnet_ref.forward(sd, x[1:2])
    net.check()
    assert (bon1.cpu() - rbon).abs().max().item() < 1e-4
    assert (cor1.cpu() - rcor).abs().max().item() < 1e-4
    # shard invariance (SURVEY 8e): a panorama's result does not depend on its batch
    assert torch.equal(bon3[1:2], bon1) and torch.equal(cor3[1:2], cor1)


def test_forward_bs32_rows_equal_bs1_bitwise_and_match_oracle():
    """The BENCHMARKED configuration (BASELINE configs[1]: batch 32, tensor cores): tile selection at B=32 differs from
    the small-batch tests (narrow tiles, whole-image row boxes, two column groups per LSTM cluster), so check it
    directly: rows {0, 13, 31} of the batch-32 forward are bit-equal to their batch-1 forwards and within 1e-4 of the CPU
    oracle (SURVEY 8d config 2)."""
    sd = synthetic_state_dict(0, 'random')           # the bench's weights
    net = _net(sd, True)
    x = synthetic_panoramas(32, seed=1000)           # the bench's first batch
    with torch.no_grad():
        bon32, cor32 = net(x.to(DEV))
    net.check()
    assert torch.isfinite(bon32).all() and torch.isfinite(cor32).all()
    for r in (0, 13, 31):
        with torch.no_grad():
            b1, c1 = net(x[r:r + 1].to(DEV))
            rb, rc = horizonnet_ref.forward(sd, x[r:r + 1])
        assert torch.equal(bon32[r:r + 1], b1) and torch.equal(cor32[r:r + 1], c1), r
        assert (b1.cpu() - rb).abs().max().item() < 1e-4, r
        assert (c1.cpu() - rc).abs().max().item() < 1e-4, r


def test_forward_pipelined_is_bitwise_equal_to_forward():
    """hn_model_forward_async (encoder of batch i+1 overlapping the bi-LSTM of batch i on internal streams) must give
    exactly the plain forward's results, for a stream of batches of different sizes, mixed with plain calls."""
    sd = synthetic_state_dict(3, 'random')
    net = _net(sd, True)
    xs = [synthetic_panoramas(b, seed=50 + i).to(DEV) for i, b in enumerate((2, 3, 1, 2))]
    with torch.no_grad():
        ref = [net(x) for x in xs]
        outs = [net.forward_pipelined(x) for x in xs]
        net.flush()
        torch.cuda.synchronize()
        for (rb, rc), (ob, oc) in zip(ref, outs):
            assert torch.equal(rb, ob) and torch.equal(rc, oc)
        # plain forward right after pipelined calls (joins the internal streams), then pipelined again
        o1 = net.forward_pipelined(xs[0])
        p2 = net(xs[1])
        o3 = net.forward_pipelined(xs[2])
        net.flush()
        torch.cuda.synchronize()
    net.check()
    assert torch.equal(o1[0], ref[0][0]) and torch.equal(p2[0], ref[1][0]) and torch.equal(o3[1], ref[2][1])


def test_nccl_gather_of_real_forward_outputs_world1():
    """SURVEY 8d config 4 on NCCL: gather_outputs (all_gather_into_tensor into preallocated buffers) returns, bit for
    bit, what the local forward produced.  One rank (the -m gpu box has one GPU); bench.py --gpus N repeats the check
    across N ranks (config.selfcheck) and the gloo world-2 tests cover the multi-rank ordering."""
    import torch.distributed as dist
    from horizonnet_b200.parallel import gather_outputs
    if dist.is_initialized():
        pytest.skip('a process group already exists in this process')
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    os.environ.setdefault('MASTER_PORT', '29533')
    dist.init_process_group('nccl', rank=0, world_size=1, device_id=torch.device(DEV))
    try:
        sd = synthetic_state_dict(1, 'random')
        net = _net(sd, True)
        x = synthetic_panoramas(2, seed=61).to(DEV)
        with torch.no_grad():
            bon, cor = net(x)
            gb, gc = gather_outputs(bon, cor)
            pb, pc = net.forward_pipelined(x)
            net.flush()
            hb, hc = gather_outputs(pb, pc)
        torch.cuda.synchronize()
        assert torch.equal(gb, bon) and torch.equal(gc, cor)
        assert torch.equal(hb, bon) and torch.equal(hc, cor)
    finally:
        dist.destroy_process_group()


def test_forward_on_does_not_switch_the_current_device():
    """ADVICE round 1: the C entry points restore the caller's current device."""
    import ctypes
    sd = synthetic_state_dict(2, 'identity')
    net = _net(sd, True)
    with torch.no_grad():
        net(synthetic_panoramas(1, seed=2).to(DEV))
    assert torch.cuda.current_device() == 0
    assert _lib.lib().hn_build_digest().decode() == __import__('horizonnet_b200.build', fromlist=['x']).source_digest()


def test_fused_bottleneck_kernel_is_bitwise_equal_to_the_unfused_convs():
    """bott_tc_kernel (layer1: conv2 + BN + ReLU -> shared memory -> conv3 + BN + identity + ReLU in one kernel) performs
    the same products in the same order with the same accumulator structure and epilogue arithmetic as conv_tc_kernel<64> +
    gemm_tc_kernel, so layer1 and the final outputs must not change by a single bit (B = 3: odd tile counts per CTA)."""
    sd = synthetic_state_dict(8, 'random')
    net = _net(sd, True)
    x = synthetic_panoramas(3, seed=71).to(DEV)
    got = {}
    with torch.no_grad():
        net(x)                                  # creates the handle
        for mode in (1, 0):
            net.set_option('fuse_bottleneck', mode)
            bon, cor = net(x)
            got[mode] = (bon.clone(), cor.clone(), net.debug_stage('layer1').clone())
        net.set_option('fuse_bottleneck', 1)
    net.check()
    assert torch.isfinite(got[1][2]).all()
    assert torch.equal(got[1][2], got[0][2]), (got[1][2] - got[0][2]).abs().max().item()
    assert torch.equal(got[1][0], got[0][0]) and torch.equal(got[1][1], got[0][1])


def test_tensor_core_stem_vs_oracle_and_fp32_stem():
    """stem_tc_kernel (7x7 s2 conv as an implicit GEMM over packed pixel pairs) against the oracle's stem in fp64
    and against the exact fp32 CUDA-core stem_kernel it replaces on the tensor-core path."""
    import torch.nn.functional as F
    sd = synthetic_state_dict(5, 'random')
    net = _net(sd, True)
    x = synthetic_panoramas(2, seed=33, channels=4)
    e = 'feature_extractor.encoder.'
    sd64 = {k: v.double() for k, v in sd.items() if k.startswith(e + 'conv1') or k.startswith(e + 'bn1.')}
    xn = (x[:, :3].double() - torch.tensor(horizonnet_ref.X_MEAN).double().view(1, 3, 1, 1)) / \
        torch.tensor(horizonnet_ref.X_STD).double().view(1, 3, 1, 1)
    ref = F.relu(horizonnet_ref._bn(horizonnet_ref._circ_conv(xn, sd64[e + 'conv1.1.weight'], None, 2, 3, 3), sd64, e + 'bn1'))
    scale = ref.abs().max().item()
    got = {}
    for mode in (1, 0):
        with torch.no_grad():
            net(x.to(DEV))                      # creates the handle on first use
            net.set_option('stem_tc', mode)
            bon, cor = net(x.to(DEV))
        net.check()
        stem = net.debug_stage('stem').cpu()
        assert tuple(stem.shape) == (2, 64, 256, 512)
        err = (stem.double() - ref).abs().max().item()
        # split-precision products carry 22 significant bits per operand (measured 5.2e-6 at scale 3.3); fp32 FMA: 1.9e-6
        assert err <= (4e-6 if mode else 1e-6) * scale + 1e-6, (mode, err, scale)
        got[mode] = (stem, bon.cpu(), cor.cpu())
    assert (got[1][1] - got[0][1]).abs().max().item() < 2e-5
    assert (got[1][2] - got[0][2]).abs().max().item() < 2e-5


def test_forward_host_equals_device_forward():
    sd = synthetic_state_dict(2, 'identity')
    net = _net(sd, True)
    x = synthetic_panoramas(2, seed=9)
    with torch.no_grad():
        bon, cor = net(x.to(DEV))
    hb, hc = net.forward_host(x.pin_memory())
    assert torch.equal(hb, bon.cpu()) and torch.equal(hc, cor.cpu())
    # pipelined host API: two batches in flight, results in submission order
    x2 = synthetic_panoramas(1, seed=10)
    with torch.no_grad():
        bon2, cor2 = net(x2.to(DEV))
    net.submit_host(x.pin_memory())
    net.submit_host(x2.pin_memory())
    pb, pc = net.collect_host()
    qb, qc = net.collect_host()
    assert torch.equal(pb, bon.cpu()) and torch.equal(pc, cor.cpu())
    assert torch.equal(qb, bon2.cpu()) and torch.equal(qc, cor2.cpu())


def test_zero_head_weight_gives_bias_exactly():
    """Known answer (SURVEY 8c): linear.weight = 0 => cor = -1, bon = (-0.478, 0.425)."""
    sd = synthetic_state_dict(4, 'identity')
    sd['linear.weight'] = torch.zeros_like(sd['linear.weight'])
    net = _net(sd, True)
    with torch.no_grad():
        bon, cor = net(synthetic_panoramas(1, seed=3).to(DEV))
    assert torch.all(cor == -1.0)
    assert torch.all(bon[:, 0] == torch.tensor(-0.478)) and torch.all(bon[:, 1] == torch.tensor(0.425))


def test_forward_rejects_wrong_size_and_reloads_weights():
    sd = synthetic_state_dict(5, 'identity')
    net = _net(sd, True)
    with pytest.raises(NotImplementedError):
        net(torch.zeros(1, 3, 256, 512, device=DEV))
    x = synthetic_panoramas(1, seed=1).to(DEV)
    with torch.no_grad():
        b0, _ = net(x)
        net.load_state_dict(synthetic_state_dict(6, 'identity'))       # in-place update must be picked up
        b1, _ = net(x)
    assert not torch.equal(b0, b1)


# ------------------------------------------------------------------------------- device-side TTA (next row f2)
def test_tta_forward_matches_reference_golden_and_oracle(golden_dir):
    from horizonnet_b200.inference import tta_forward
    from oracle import tta_ref
    g = np.load(os.path.join(golden_dir, 'tta_randombn.npz'))
    sd = synthetic_state_dict(int(g['seed']), 'random')
    net = _net(sd, True)
    x = synthetic_panoramas(1, seed=int(g['x_seed']))
    y_bon, y_cor = tta_forward(net, x, flip=bool(g['flip']), rotate=list(g['rotate']))
    assert y_bon.shape == (2, 1024) and y_cor.shape == (1024,)
    # boundary rows in pixels: 1e-4 rad * 512/pi = 1.6e-2 px is the forward tolerance; cor: sigmoid of 1e-4
    assert np.abs(y_bon - g['y_bon']).max() < 1.6e-2
    assert np.abs(y_cor - g['y_cor']).max() < 1e-4
    # no-augmentation path == plain forward + decode, and oracle agreement on another setting
    y_bon0, y_cor0 = tta_forward(net, x)
    with torch.no_grad():
        bon, cor = net(x.to(DEV))
    ref_rows = (bon[0].cpu().numpy() / np.float32(np.pi) + 0.5) * 512 - 0.5
    ref_rows[0] = np.clip(ref_rows[0], 1, 255); ref_rows[1] = np.clip(ref_rows[1], 257, 510)
    assert np.abs(y_bon0 - ref_rows).max() < 1e-3
    assert np.abs(y_cor0 - torch.sigmoid(cor[0, 0]).cpu().numpy()).max() < 1e-6
    ob, oc = tta_ref.tta_forward(sd, x, flip=False, rotate=[0.5])
    tb, tc = tta_forward(net, x, flip=False, rotate=[0.5])
    assert np.abs(tb - ob).max() < 1.6e-2 and np.abs(tc - oc).max() < 1e-4


# ------------------------------------------------------------------------------- pano_stretch
def test_pano_stretch_small_grid_vs_golden(golden_dir):
    g = dict(np.load(os.path.join(golden_dir, 'panostretch_small.npz')))
    g.update(np.load(os.path.join(golden_dir, 'panostretch_small_kx_above_1.npz')))
    img = g['img']
    for kx in KGRID:
        for ky in KGRID:
            out, _ = pano_stretch(img, np.zeros((1, 2), np.float32), kx, ky)
            assert out.dtype == np.float32 and out.shape == img.shape
            assert np.abs(out - g[f'out_{kx}_{ky}']).max() <= 1.2e-7, (kx, ky)
    out0, _ = pano_stretch(img, np.zeros((1, 2), np.float32), 1.5, 0.75, order=0)
    assert np.mean(out0 != g['out0_1.5_0.75']) < 1e-3          # nearest: ties may round differently


def test_pano_stretch_full_size_vs_golden_and_oracle(golden_dir):
    g = np.load(os.path.join(golden_dir, 'panostretch_rows.npz'))
    img = np.random.RandomState(0).random_sample((512, 1024, 3)).astype(np.float32)
    corners = np.array([[158, 186], [158, 329], [353, 185], [353, 330], [594, 154], [594, 363],
                        [713, 100], [713, 415], [692, 77], [692, 438], [965, 150], [965, 367]], np.float32)
    rows = g['rows']
    pairs = [(kx, ky) for kx in KGRID for ky in KGRID]
    dev_img = torch.from_numpy(img).to(DEV)
    batch = dev_img.unsqueeze(0).expand(len(pairs), -1, -1, -1).contiguous()
    outs = pano_stretch_batch(batch, [p[0] for p in pairs], [p[1] for p in pairs]).cpu().numpy()
    for i, (kx, ky) in enumerate(pairs):
        o = outs[i]
        assert abs(o.astype(np.float64).sum() - float(g[f'sum_{kx}_{ky}'])) < 1e-3 * 1.0, (kx, ky)
        assert abs((o.astype(np.float64) ** 2).sum() - float(g[f'sq_{kx}_{ky}'])) < 1e-3, (kx, ky)
        if f'out_{kx}_{ky}' in g.files:
            assert np.abs(o[rows] - g[f'out_{kx}_{ky}']).max() <= 1.2e-7, (kx, ky)
    # one full image against the oracle, plus the host (numpy) entry point and corners
    out, cor = pano_stretch(img, corners, 2.0, 0.5)
    rout, rcor = panostretch_ref.pano_stretch(img, corners, 2.0, 0.5)
    assert np.abs(out - rout).max() <= 1.2e-7
    assert np.abs(cor - rcor).max() < 1e-9 and cor.dtype == rcor.dtype
    assert np.array_equal(out, outs[pairs.index((2.0, 0.5))])
    # identity (SURVEY 8c)
    ident, icor = pano_stretch(img, corners, 1.0, 1.0)
    assert np.abs(ident - img).max() <= 1.2e-7 and np.abs(icor - corners).max() < 1e-4


@pytest.mark.parametrize('shape', [(7, 10, 1), (33, 130, 3), (64, 258, 4), (1, 8, 2), (2, 8, 2)])
def test_pano_stretch_ragged_shapes_vs_oracle(shape):
    img = np.random.RandomState(sum(shape)).random_sample(shape).astype(np.float32)
    for kx, ky in ((0.6, 1.9), (1.8, 0.7), (1.0, 1.0)):
        out, _ = pano_stretch(img, np.zeros((1, 2)), kx, ky)
        rout, _ = panostretch_ref.pano_stretch(img, np.zeros((1, 2)), kx, ky)
        assert np.abs(out - rout).max() <= 1.2e-7, (shape, kx, ky, out.ravel()[:8], rout.ravel()[:8])


def test_pano_stretch_float64_images_like_the_reference_cli():
    """misc/panostretch.py:171 feeds float64 0-255 images: scipy then interpolates and returns float64; so do we."""
    img = (np.random.RandomState(4).random_sample((40, 96, 3)) * 255.0)
    assert img.dtype == np.float64
    for kx, ky in ((2.0, 1.0), (0.6, 1.7)):
        out, _ = pano_stretch(img, np.zeros((1, 2)), kx, ky)
        rout, _ = panostretch_ref.pano_stretch(img, np.zeros((1, 2)), kx, ky)
        assert out.dtype == np.float64 and np.abs(out - rout).max() <= 1e-10, (kx, ky, np.abs(out - rout).max())


def test_pano_stretch_rejects_bad_arguments():
    with pytest.raises(TypeError):
        pano_stretch(np.zeros((8, 16, 3), np.uint8), np.zeros((1, 2)), 1.0, 1.0)
    with pytest.raises(RuntimeError):
        pano_stretch(np.zeros((8, 16, 3), np.float32), np.zeros((1, 2)), -1.0, 1.0)
    empty = pano_stretch_batch(torch.zeros(0, 8, 16, 3, device=DEV), [], [])
    assert empty.shape == (0, 8, 16, 3)


# ------------------------------------------------------------------------------- "next" row f3: fused augmentation
def _synthetic_u8(h, w, seed):
    return np.random.RandomState(seed).randint(0, 256, size=(h, w, 3)).astype(np.uint8)


def test_augment_matches_the_real_dataset_pipeline_golden(golden_dir):
    """hn_augment (uint8 HWC -> stretch -> flip -> roll -> gamma -> float32 CHW in one pass) against the tensor the
    REAL dataset.PanoCorBonDataset.__getitem__ produced (tests/golden/augment.npz).  Tolerance 3e-7: one fp32 ulp of the
    bilinear result (1.2e-7, as for pano_stretch) carried through x**p plus CUDA powf vs numpy's float32 power (a few ulp)."""
    from horizonnet_b200.augment import augment_batch
    g = np.load(os.path.join(golden_dir, 'augment.npz'))
    for c in range(int(g['n_cases'])):
        h, w = (int(v) for v in g[f'c{c}_hw'])
        kx, ky, flip, dx, p = (float(v) for v in g[f'c{c}_params'])
        img = _synthetic_u8(h, w, int(g[f'c{c}_img_seed']))
        x = augment_batch(img[None], [kx], [ky], [bool(flip)], [int(dx)], [p])[0].cpu().numpy()
        assert x.shape == (3, h, w) and x.dtype == np.float32
        got = x if h < 512 else x[:, g['rows']]
        assert np.abs(got - g[f'c{c}_x']).max() <= 3e-7, (c, np.abs(got - g[f'c{c}_x']).max())
        assert abs(x.astype(np.float64).sum() - float(g[f'c{c}_sum'])) < 0.05, c


def test_augment_option_combinations_vs_oracle():
    """Every on/off combination of the four augmentations (per image, in one batch) against oracle/augment_ref.py; without
    gamma the result is the float32 bilinear value itself: 1.2e-7 like pano_stretch; identity = uint8 / 255 exactly."""
    from horizonnet_b200.augment import augment_batch
    from oracle import augment_ref
    h, w = 48, 96
    imgs = np.stack([_synthetic_u8(h, w, 70 + i) for i in range(16)])
    rs = np.random.RandomState(9)
    kx, ky, flip, dx, gam = [], [], [], [], []
    for i in range(16):
        st = bool(i & 1)
        kx.append(float(rs.uniform(0.5, 2.0)) if st else None); ky.append(float(rs.uniform(0.5, 2.0)) if st else None)
        flip.append(bool(i & 2)); dx.append(int(rs.randint(w)) if i & 4 else 0)
        gam.append(float(rs.uniform(0.5, 2.0)) if i & 8 else None)
    x = augment_batch(imgs, kx, ky, flip, dx, gam).cpu().numpy()
    for i in range(16):
        ref = augment_ref.augment_image(imgs[i], kx[i], ky[i], flip[i], dx[i], gam[i])
        tol = 3e-7 if gam[i] is not None else 1.2e-7
        assert np.abs(x[i] - ref).max() <= tol, (i, np.abs(x[i] - ref).max())
    assert np.array_equal(x[0], (imgs[0].astype(np.float32) / np.float32(255.)).transpose(2, 0, 1))
    with pytest.raises(RuntimeError):
        augment_batch(imgs[:1], dx=[w])                       # dx out of range (np.random.randint(W) never yields W)
    with pytest.raises(TypeError):
        augment_batch(imgs[:1].astype(np.float32))


# ------------------------------------------------------------------------------- "next" row f4: rotatePanorama
def test_rotate_panorama_matches_the_real_reference_golden(golden_dir):
    from horizonnet_b200.misc.pano_lsd_align import rotatePanorama, rotate_panorama_batch
    from oracle import panorotate_ref
    g = np.load(os.path.join(golden_dir, 'rotate.npz'))
    out = rotatePanorama(g['small_img'], R=g['small_R'])
    assert out.dtype == np.float64 and out.shape == g['small_out'].shape
    assert np.abs(out - g['small_out']).max() < 1e-12
    assert np.abs(rotatePanorama(g['small_img'], g['small_R'][2::-1]) - g['small_out_vp']).max() < 1e-12
    img = np.random.RandomState(22).random_sample((512, 1024, 3)).astype(np.float32)
    batch = torch.from_numpy(img).to(DEV).unsqueeze(0)
    for name in ('tilt', 'big'):
        o = rotate_panorama_batch(batch, R=g[f'{name}_R'])[0].cpu().numpy()
        assert np.abs(o[g["rows"]] - g[f"{name}_rows"]).max() < 1e-10, name   # R^-1 product vs the reference's per-pixel LU solve
        assert abs(o.sum() - float(g[f'{name}_sum'])) < 1e-6 and abs((o ** 2).sum() - float(g[f'{name}_sq'])) < 1e-6, name
    # identity rotation reproduces the image (the padding never contributes); odd sizes / 1 channel vs the oracle
    ident = rotatePanorama(g['small_img'], R=np.eye(3))
    assert np.abs(ident - g['small_img']).max() < 1e-12
    img1 = np.random.RandomState(5).random_sample((17, 30, 1))
    q, _ = np.linalg.qr(np.random.RandomState(6).randn(3, 3))
    assert np.abs(rotatePanorama(img1, R=q) - panorotate_ref.rotate_panorama(img1, R=q)).max() < 1e-12
    with pytest.raises(RuntimeError):
        rotatePanorama(np.zeros((8, 15, 3)), R=np.eye(3))         # odd width: the reference's padding rule is undefined


# ------------------------------------------------------------------------------- train-mode forward (row f1, forward only)
def _train_net(sd, tensor_cores, frozen=(), momentum=None):
    net = HorizonNet('resnet50', True)
    net.load_state_dict(sd, strict=True)
    net.use_tensor_cores(tensor_cores)
    net = net.to(DEV).train()                                           # train.py:249
    if frozen:                                                          # train.py:251-256 (--freeze_earlier_blocks 1)
        blocks = net.feature_extractor.list_blocks()
        for i in range(2):
            for m in blocks[i]:
                m.eval()
        assert sorted(n for n, m in net.named_modules() if isinstance(m, torch.nn.BatchNorm2d) and not m.training) == \
            sorted(frozen)
    if momentum is not None:
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.momentum = momentum                                   # train.py:210-213
    return net


@pytest.mark.parametrize('tensor_cores', [False, True])
@pytest.mark.parametrize('name', ['all', 'frozen1'])
def test_train_forward_matches_the_real_reference_golden(golden_dir, name, tensor_cores):
    """net.train(); net(x) (train.py:52) against the REAL reference's train-mode forward: batch-statistics BatchNorm,
    running-statistics update, both dropouts (the reference's own masks, injected), frozen blocks and --bn_momentum."""
    from train_fixture import train_golden
    g, sd, x, masks, running, frozen = train_golden(golden_dir, name)
    net = _train_net(sd, tensor_cores, frozen, float(g['momentum']) if name == 'frozen1' else None)
    net.dropout_masks_override = masks
    with torch.no_grad():                        # no tape: the tensor-core / fp32 inference kernels, each conv twice
        bon, cor = net(x.to(DEV))
    net.check()
    assert np.abs(bon.cpu().numpy() - g['bon']).max() < 1e-4
    assert np.abs(cor.cpu().numpy() - g['cor']).max() < 1e-4
    assert not bon.requires_grad
    after = net.state_dict()
    for k, v in running.items():
        if k.rsplit('.', 1)[0] in frozen:
            assert torch.equal(after[k].cpu(), sd[k]), k
        else:
            assert torch.allclose(after[k].cpu(), v, rtol=1e-4, atol=1e-5), k
    nbt = [int(after[k]) for k in after if k.endswith('num_batches_tracked')]
    assert nbt == list(g['num_batches_tracked'])
    # back to eval: the moved running statistics are the ones folded into the inference graph now
    net.eval()
    after_cpu = {k: v.cpu() for k, v in after.items()}
    with torch.no_grad():
        ebon, ecor = net(x[:1].to(DEV))
        rbon, rcor = horizonnet_ref.forward(after_cpu, x[:1])
    assert (ebon.cpu() - rbon).abs().max().item() < 1e-4 and (ecor.cpu() - rcor).abs().max().item() < 1e-4
    with torch.no_grad():
        obon, _ = horizonnet_ref.forward(sd, x[:1])
    assert (rbon - obon).abs().max().item() > 1e-3 or name == 'frozen1'     # ... and they did move the result


def test_train_forward_with_device_dropout_masks_matches_oracle_and_is_seeded():
    """The library's own Philox masks: a pure function of the seed (drawn from torch's generator, so torch.manual_seed
    makes a run reproducible), Bernoulli(0.5) scaled by 2, independent between the two dropouts; the oracle fed with
    exactly those masks agrees with the device forward."""
    sd = synthetic_state_dict(5, 'random')
    x = synthetic_panoramas(2, seed=31)
    net = _train_net(sd, True)
    torch.manual_seed(77)
    with torch.no_grad():
        bon, cor = net(x.to(DEV))
    seed = net.last_dropout_seed
    m0, m1 = net.dropout_masks(seed, 2, DEV)
    for m in (m0, m1):
        assert set(torch.unique(m).tolist()) == {0.0, 2.0}
        assert abs(float((m > 0).float().mean()) - 0.5) < 0.005
    assert 0.45 < float(((m0 > 0) == (m1 > 0)).float().mean()) < 0.55
    tm = horizonnet_ref.TrainMode(masks=[m0.cpu(), m1.cpu()])
    with torch.no_grad():
        rbon, rcor = horizonnet_ref.forward(sd, x, train=tm)
    assert (bon.cpu() - rbon).abs().max().item() < 1e-4 and (cor.cpu() - rcor).abs().max().item() < 1e-4
    # same torch seed, fresh weights -> same masks -> bit-identical outputs; another seed -> other masks
    net2 = _train_net(sd, True)
    torch.manual_seed(77)
    with torch.no_grad():
        bon2, cor2 = net2(x.to(DEV))
        bon3, _ = net2(x.to(DEV))
    assert net2.last_dropout_seed != seed and torch.equal(bon2, bon) and torch.equal(cor2, cor)
    assert not torch.equal(bon3, bon)
    # dropout off (p = 0 modules in eval) but BatchNorm in train mode: still the train path, no masks
    net2.bi_rnn.eval(); net2.drop_out.eval()
    assert net2._train_mode_active()
    net3 = _train_net(sd, True)
    net3.bi_rnn.eval(); net3.drop_out.eval()
    with torch.no_grad():
        b3, c3 = net3(x.to(DEV))
    tm = horizonnet_ref.TrainMode(p=0.0)
    with torch.no_grad():
        rb, rc = horizonnet_ref.forward(sd, x, train=tm)
    assert (b3.cpu() - rb).abs().max().item() < 1e-4 and (c3.cpu() - rc).abs().max().item() < 1e-4


# ------------------------------------------------------------------------------- training step: backward (row f1)
BWD_CONV_CASES = [
    # B, Cin, H, W, Cout, k, stride, in_halo, data gradient?
    (2, 32, 8, 16, 48, 3, (1, 1), 1, True),
    (2, 64, 8, 16, 64, 1, (1, 1), 1, True),
    (1, 64, 8, 16, 32, 3, (2, 2), 1, True),        # layer2-4 conv2 of the first block
    (2, 128, 4, 16, 64, 1, (2, 2), 1, True),       # downsample
    (2, 64, 8, 16, 32, 3, (2, 1), 1, True),        # height-reduction conv
    (3, 16, 6, 62, 48, 3, (1, 1), 1, True),        # ragged: Cout % 64 != 0, K % 64 != 0, M not a multiple of 16*slices
    (1, 3, 16, 32, 64, 7, (2, 2), 3, False),       # stem: weight gradient only, Cin = 3
    (2, 512, 2, 32, 256, 3, (2, 1), 1, True),      # real height-reduction shapes: H 2 -> 1
    (2, 64, 16, 256, 32, 3, (2, 1), 1, True),      # ghc_lst.0.layer.3: W = 256, Cout = 32, several pixel slices
    (2, 1024, 4, 32, 512, 3, (2, 1), 1, True),     # ghc_lst.3.layer.2: K = 9216
    (2, 128, 16, 64, 192, 3, (1, 1), 1, False),    # 128 x 128 weight-gradient tile with a ragged second tile (Cout = 192, K = 1152)
    (3, 256, 10, 32, 128, 1, (1, 1), 1, True),     # 1x1, K = 256: two full k tiles, M = 960 over several slices
]


@pytest.mark.parametrize('case', BWD_CONV_CASES)
def test_conv_backward_vs_autograd(case):
    """Weight gradient (conv_wgrad_f32) and data gradient (forward conv kernel on the dilated output gradient with
    flipped weights) of one circular-W convolution against torch.autograd in fp64."""
    B, Ci, H, W, Co, k, stride, in_halo, want_din = case
    g = torch.Generator().manual_seed(hash(case) % (2 ** 31))
    x = torch.randn(B, Ci, H, W, generator=g)
    w = torch.randn(Co, Ci, k, k, generator=g) / (Ci * k * k) ** 0.5
    p = k // 2
    xd = x.double().requires_grad_()
    wd = w.double().requires_grad_()
    xp = torch.cat([xd[..., -p:], xd, xd[..., :p]], dim=3) if p else xd
    y = torch.nn.functional.conv2d(xp, wd, None, stride=stride, padding=(p, 0))
    dz = torch.randn(y.shape, generator=g)
    y.backward(dz.double())
    lib = _lib.lib()
    xin = gu.to_halo_nhwc(x, in_halo).to(DEV)
    dzin = gu.to_halo_nhwc(dz, 1).to(DEV)
    wdev = w.to(DEV)
    dw = torch.full_like(wdev, float('nan'))
    din = torch.full((B, H, W + 2, Ci), float('nan'), device=DEV) if want_din else None
    _lib.check(lib.hn_conv2d_backward(xin.data_ptr(), B, H, W, Ci, in_halo, wdev.data_ptr(), dzin.data_ptr(), Co, k, k,
                                      stride[0], stride[1], p, p, din.data_ptr() if want_din else None, dw.data_ptr(),
                                      torch.cuda.current_stream().cuda_stream), 'hn_conv2d_backward')
    torch.cuda.synchronize()
    ref_w = wd.grad
    assert (dw.cpu().double() - ref_w).abs().max().item() <= 2e-5 * ref_w.abs().max().item()
    if want_din:
        got = gu.from_halo_nhwc(din, 1).cpu().double()
        assert (got - xd.grad).abs().max().item() <= 2e-5 * xd.grad.abs().max().item()


WGRAD_TC_CASES = [
    # B, Cin, H, W, Cout, k, stride        (Cin, Cout multiples of 64; the tile shapes of the real units)
    (2, 64, 8, 256, 64, 3, (1, 1)),        # layer1 conv2: one 64-channel atom on both sides, half rows (W = 256 -> 4 tiles per row)
    (2, 256, 8, 256, 64, 1, (1, 1)),       # layer1 conv1: two Cin tiles
    (2, 64, 8, 256, 256, 1, (1, 1)),       # layer1 conv3 / downsample: two Cout tiles
    (2, 128, 8, 128, 128, 3, (2, 2)),      # layer2.0 conv2: stride 2 both ways (parity view + row traversal stride)
    (2, 256, 8, 128, 512, 1, (2, 2)),      # layer2.0 downsample
    (2, 256, 16, 256, 128, 3, (2, 1)),     # ghc_lst.0.layer.0: stride (2, 1), W = 256
    (2, 128, 4, 64, 128, 3, (1, 1)),       # layer3-like: W = 64, one row per tile
    (2, 192, 8, 32, 192, 3, (1, 1)),       # W = 32: two rows per tile; second channel tile has one atom on both sides
    (3, 512, 2, 32, 256, 3, (2, 1)),       # ghc_lst.3.layer.3: H 2 -> 1, two images per tile, ragged last tile (B = 3)
    (5, 64, 2, 16, 128, 3, (2, 1)),        # W = 16: four images per tile, B = 5
    (2, 1024, 4, 32, 512, 3, (2, 1)),      # ghc_lst.3.layer.2: 8 x 4 channel tiles, 9 taps
    (4, 128, 32, 64, 128, 3, (1, 1)),      # 8192 pixels = 128 tiles: more than one pixel slice per work item
]


def _record(name, payload):
    """Measured errors of the new kernels, kept next to the gpurun logs when that directory exists."""
    import json
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'gpurun_out')
    if os.path.isdir(d):
        with open(os.path.join(d, name), 'a') as f:
            f.write(json.dumps(payload) + '\n')


@pytest.mark.parametrize('case', WGRAD_TC_CASES)
def test_conv_wgrad_tc_vs_autograd(case):
    """Weight gradient on the tcgen05 kernel (wgrad_tc.cu: pixel-axis GEMM over MN-major plane tiles) against
    torch.autograd in fp64, and against the fp32 CUDA-core kernel on the same inputs."""
    B, Ci, H, W, Co, k, stride = case
    g = torch.Generator().manual_seed(hash(case) % (2 ** 31))
    x = torch.randn(B, Ci, H, W, generator=g)
    p = k // 2
    wd = (torch.randn(Co, Ci, k, k, generator=g, dtype=torch.float64) / (Ci * k * k) ** 0.5).requires_grad_()
    xd = x.double()
    xp = torch.cat([xd[..., -p:], xd, xd[..., :p]], dim=3) if p else xd
    y = torch.nn.functional.conv2d(xp, wd, None, stride=stride, padding=(p, 0))
    dz = torch.randn(y.shape, generator=g) * 1e-4          # gradients are small: the planes carry a power-of-two scale
    y.backward(dz.double())
    lib = _lib.lib()
    xin = gu.to_halo_nhwc(x, 1).to(DEV)
    dzin = gu.to_halo_nhwc(dz, 1).to(DEV)
    st = torch.cuda.current_stream().cuda_stream
    dw = torch.full((Co, Ci, k, k), float('nan'), device=DEV)
    _lib.check(lib.hn_conv2d_wgrad_tc(xin.data_ptr(), B, H, W, Ci, dzin.data_ptr(), Co, k, k, stride[0], stride[1], p, p,
                                      dw.data_ptr(), st), 'hn_conv2d_wgrad_tc')
    dw32 = torch.full_like(dw, float('nan'))
    wdev = wd.detach().float().to(DEV)
    _lib.check(lib.hn_conv2d_backward(xin.data_ptr(), B, H, W, Ci, 1, wdev.data_ptr(), dzin.data_ptr(), Co, k, k,
                                      stride[0], stride[1], p, p, None, dw32.data_ptr(), st), 'hn_conv2d_backward')
    torch.cuda.synchronize()
    ref = wd.grad
    scale = ref.abs().max().item()
    err = (dw.cpu().double() - ref).abs().max().item() / scale
    err32 = (dw32.cpu().double() - ref).abs().max().item() / scale
    _record('wgrad_tc_errors.jsonl', {'case': list(case[:6]) + list(stride), 'err_tc': err, 'err_fp32': err32,
                                      'desc': os.environ.get('HN_WGRAD_TC_DESC', '0')})
    assert err <= 2e-5, (err, err32)


def test_conv_wgrad_tc_rejects_shapes_it_does_not_take():
    lib = _lib.lib()
    x = torch.zeros(1, 8, 18, 48, device=DEV)
    dz = torch.zeros(1, 8, 18, 64, device=DEV)
    dw = torch.zeros(64, 48, 3, 3, device=DEV)
    assert lib.hn_conv2d_wgrad_tc(x.data_ptr(), 1, 8, 16, 48, dz.data_ptr(), 64, 3, 3, 1, 1, 1, 1, dw.data_ptr(), None) != 0
    assert b'not supported' in _lib.lib().hn_last_error()


def test_training_step_weight_gradients_tcgen05_vs_fp32_kernels(monkeypatch):
    """The whole backward of one batch-2 step with the weight gradients on the tcgen05 kernel (HN_WGRAD_TC=1) against the
    same step with the fp32 CUDA-core weight-gradient kernel (=0): same tape, same dz, so every parameter gradient
    agrees to rounding."""
    import torch.nn.functional as F
    sd = synthetic_state_dict(5, 'random')
    x = synthetic_panoramas(2, seed=53).to(DEV)
    y_bon, y_cor = torch.zeros(2, 2, 1024, device=DEV), torch.full((2, 1, 1024), 0.5, device=DEV)
    grads = {}
    for mode in ('0', '1'):
        monkeypatch.setenv('HN_WGRAD_TC', mode)
        assert _lib.lib().hn_wgrad_tc_enabled() == int(mode)
        net = _train_net(sd, True)
        torch.manual_seed(3)
        bon, cor = net(x)
        (F.l1_loss(bon, y_bon) + F.binary_cross_entropy_with_logits(cor, y_cor)).backward()
        net.check()
        grads[mode] = {k: p.grad.clone() for k, p in net.named_parameters()}
    gmax = max(float(v.abs().max()) for v in grads['0'].values())
    worst = sorted(((float((grads['1'][k] - v).abs().max()) / (float(v.abs().max()) + 1e-4 * gmax), k)
                    for k, v in grads['0'].items()), reverse=True)
    _record('wgrad_tc_errors.jsonl', {'whole_step_worst': worst[:5]})
    assert worst[0][0] < 1e-4, worst[:8]


@pytest.mark.parametrize('shape', [(3, 32, 5, 8), (2, 256, 4, 70), (2, 96, 3, 33)])
@pytest.mark.parametrize('train,relu,res', [(1, 1, True), (1, 0, False), (0, 1, True), (1, 1, False)])
def test_batchnorm_forward_backward_vs_autograd(train, relu, res, shape):
    B, C, H, W = shape          # channel-quad lanes x pixel lanes of the reduction kernels: 8 x 32, 64 x 4, 16 x 16 (24 quads)
    g = torch.Generator().manual_seed(3 + train + 2 * relu)
    z = torch.randn(B, C, H, W, generator=g) * 2 + 0.5
    gamma, beta = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.1
    rm, rv = torch.randn(C, generator=g) * 0.1, torch.rand(C, generator=g) + 0.5
    r = torch.randn(B, C, H, W, generator=g) if res else None
    dy = torch.randn(B, C, H, W, generator=g)
    zd, gd, bd = z.double().requires_grad_(), gamma.double().requires_grad_(), beta.double().requires_grad_()
    rd = r.double().requires_grad_() if res else None
    rm2, rv2 = rm.double().clone(), rv.double().clone()
    y = torch.nn.functional.batch_norm(zd, rm2, rv2, gd, bd, bool(train), 0.1, 1e-5)
    if res:
        y = y + rd
    if relu:
        y = torch.relu(y)
    y.backward(dy.double())
    dev = lambda t: gu.to_halo_nhwc(t, 1).to(DEV)
    zt, dyt = dev(z), dev(dy)
    rt = dev(r) if res else None
    yt, dzt = torch.empty_like(zt), torch.full_like(zt, float('nan'))
    drt = torch.zeros_like(zt) if res else None
    gam, bet, rmt, rvt = gamma.to(DEV), beta.to(DEV), rm.to(DEV), rv.to(DEV)
    dgam, dbet = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
    scratch, sums = torch.empty(4 * C, device=DEV), torch.zeros(3 * C, device=DEV, dtype=torch.float64)
    _lib.check(_lib.lib().hn_bn_forward_backward(
        zt.data_ptr(), B, H, W, C, gam.data_ptr(), bet.data_ptr(), rmt.data_ptr(), rvt.data_ptr(), 0.1, train, relu,
        rt.data_ptr() if res else None, yt.data_ptr(), dyt.data_ptr(), dzt.data_ptr(), drt.data_ptr() if res else None,
        dgam.data_ptr(), dbet.data_ptr(), scratch.data_ptr(), sums.data_ptr(), torch.cuda.current_stream().cuda_stream),
        'hn_bn_forward_backward')
    torch.cuda.synchronize()
    close = lambda a, b, tol=2e-5: (a.cpu().double() - b).abs().max().item() <= tol * max(1.0, b.abs().max().item())
    assert close(gu.from_halo_nhwc(yt, 1), y.detach())
    assert torch.equal(yt[:, :, 0], yt[:, :, -2]) and torch.equal(dzt[:, :, -1], dzt[:, :, 1])      # circular halo columns
    assert close(gu.from_halo_nhwc(dzt, 1), zd.grad)
    assert close(dgam, gd.grad) and close(dbet, bd.grad)
    if res:
        assert close(gu.from_halo_nhwc(drt, 1), rd.grad)
    if train:
        assert close(rmt, rm2) and close(rvt, rv2)
    else:
        assert torch.equal(rmt.cpu(), rm) and torch.equal(rvt.cpu(), rv)


@pytest.mark.parametrize('T,B', [(6, 2), (9, 11)])
def test_lstm_layer_backward_vs_autograd(T, B):
    """Gate gradients of one bidirectional layer (recompute of the gates from the saved outputs, cell scan, one launch
    per time step) against autograd through the oracle's LSTM."""
    g = torch.Generator().manual_seed(T * 100 + B)
    x = torch.randn(T, B, 1024, generator=g) * 0.5
    ws = {}
    for sfx in ('', '_reverse'):
        ws['ih' + sfx] = (torch.randn(2048, 1024, generator=g) / 32)
        ws['hh' + sfx] = (torch.randn(2048, 512, generator=g) / 22)
        ws['b' + sfx] = torch.randn(2048, generator=g) * 0.1
    xps, outs = [], []
    for sfx, rev in (('', False), ('_reverse', True)):
        xp = (x.double() @ ws['ih' + sfx].double().t() + ws['b' + sfx].double()).requires_grad_()
        xps.append(xp)
        # the oracle's recurrence with the input projection made explicit (so that d xp is observable)
        h = torch.zeros(B, 512, dtype=torch.float64)
        c = torch.zeros(B, 512, dtype=torch.float64)
        out = [None] * T
        for t in (range(T - 1, -1, -1) if rev else range(T)):
            gt = xp[t] + h @ ws['hh' + sfx].double().t()
            i, f, gg, o = gt.chunk(4, dim=1)
            c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
            h = torch.sigmoid(o) * torch.tanh(c)
            out[t] = h
        outs.append(torch.stack(out))
    hout = torch.cat(outs, dim=2)
    dout = torch.randn(T, B, 1024, generator=g)
    hout.backward(dout.double())
    xp_all = torch.cat([xps[0].detach(), xps[1].detach()], dim=2).float().contiguous().to(DEV)
    rows = T * B
    scratch = torch.empty(2 * rows * 512 * 2 + 2 * rows * 2048 + 2 * B * 512 + 2 * 512 * 2048 + 8192, device=DEV)
    dg = torch.full((2, T, B, 2048), float('nan'), device=DEV)
    hout_d, whf, whb, dout_d = (t.detach().float().contiguous().to(DEV) for t in (hout, ws['hh'], ws['hh_reverse'], dout))
    _lib.check(_lib.lib().hn_lstm_layer_backward(
        xp_all.data_ptr(), hout_d.data_ptr(), whf.data_ptr(), whb.data_ptr(), dout_d.data_ptr(), T, B, dg.data_ptr(),
        scratch.data_ptr(), torch.cuda.current_stream().cuda_stream), 'hn_lstm_layer_backward')
    torch.cuda.synchronize()
    for d in range(2):
        ref = xps[d].grad
        assert (dg[d].cpu().double() - ref).abs().max().item() <= 5e-5 * ref.abs().max().item(), d


@pytest.mark.parametrize('tensor_cores,wgrad_tc', [(True, '1'), (True, '0'), (False, '0')])
def test_training_step_gradients_match_autograd_of_the_oracle(tensor_cores, wgrad_tc, monkeypatch):
    """tensor_cores: forward convolutions and data gradients on the tcgen05 kernel (default) / everything on the fp32
    CUDA-core kernels; wgrad_tc: weight gradients on the tcgen05 kernel where it applies (HN_WGRAD_TC).  BASELINE config 5 (train.py:44-58 + :278) at batch 2: net.train(); loss = L1(bon) + BCE-with-logits(cor);
    loss.backward() through the library against torch.autograd through the CPU oracle with the same dropout masks,
    for every one of the reference's parameters."""
    import torch.nn.functional as F
    sd = synthetic_state_dict(1, 'random')
    x = synthetic_panoramas(2, seed=41)
    gen = torch.Generator().manual_seed(9)
    y_bon = torch.rand(2, 2, 1024, generator=gen) - 0.5
    y_cor = torch.rand(2, 1, 1024, generator=gen)
    monkeypatch.setenv('HN_WGRAD_TC', wgrad_tc)
    net = _train_net(sd, tensor_cores)
    torch.manual_seed(11)
    bon, cor = net(x.to(DEV))
    assert bon.requires_grad and cor.requires_grad
    loss = F.l1_loss(bon, y_bon.to(DEV)) + F.binary_cross_entropy_with_logits(cor, y_cor.to(DEV))     # train.py:53-56
    loss.backward()                                                                                    # train.py:278
    net.check()
    masks = [t.cpu() for t in net.dropout_masks(net.last_dropout_seed, 2, DEV)]
    names = [k for k, _ in net.named_parameters()]

    def oracle_grads(relu_masks):
        psd = {k: (v.clone().requires_grad_() if k in names else v) for k, v in sd.items()}
        tm = horizonnet_ref.TrainMode(masks=masks, relu_masks=relu_masks)
        rbon, rcor = horizonnet_ref.forward(psd, x, train=tm)
        rloss = F.l1_loss(rbon, y_bon) + F.binary_cross_entropy_with_logits(rcor, y_cor)
        return rbon.detach(), rloss.item(), dict(zip(names, torch.autograd.grad(rloss, [psd[k] for k in names])))

    def worst_errors(ref):
        gmax = max(float(v.abs().max()) for v in ref.values())
        out = []
        for k, p in net.named_parameters():
            assert p.grad is not None and p.grad.shape == p.shape, k
            err = float((p.grad.cpu() - ref[k]).abs().max())
            out.append((err / (float(ref[k].abs().max()) + 1e-4 * gmax), k))    # 1e-4 * gmax: the conv biases in front of a
            # train-mode BatchNorm have an analytically zero gradient (autograd returns rounding noise there)
        return sorted(out, reverse=True)

    # (1) the oracle on its own: forward and loss agree; the gradients agree up to ReLU decisions -- the two fp32
    #     forwards differ by ~1e-4 deep in the net (train-mode BN on 2 panoramas amplifies rounding), which flips the
    #     sign of ~1 % of the near-zero pre-activations, and each flip moves a gradient element by its full value
    rbon, rloss, ref = oracle_grads(None)
    assert (bon.detach().cpu() - rbon).abs().max().item() < 1e-4
    assert abs(loss.item() - rloss) < 1e-5
    free = worst_errors(ref)
    assert free[0][0] < 0.5, free[:8]
    # (2) the same ReLU decisions on both sides (the device's, read from its tape): every gradient agrees
    relu_masks = {}
    for i in range(69):
        name, y = net.debug_train_unit(i, 0)
        if not name.endswith('downsample.1'):
            relu_masks[name] = (y > 0).cpu()
    _, rloss2, ref2 = oracle_grads(relu_masks)
    assert abs(loss.item() - rloss2) < 1e-5
    same = worst_errors(ref2)
    assert same[0][0] < 5e-3, same[:8]
    # a second step on the same handle (the tape is rebuilt; gradients accumulate into .grad like torch's do)
    g0 = net.linear.weight.grad.clone()
    bon2, cor2 = net(x.to(DEV))
    (F.l1_loss(bon2, y_bon.to(DEV)) + F.binary_cross_entropy_with_logits(cor2, y_cor.to(DEV))).backward()
    assert not torch.equal(net.linear.weight.grad, g0)


def test_training_step_with_frozen_blocks_like_freeze_earlier_blocks():
    """train.py --freeze_earlier_blocks 1 (:200-208 requires_grad = False, :251-256 those blocks in eval mode):
    frozen BatchNorm2d modules use and keep their running statistics, frozen parameters get no gradient, the rest
    agree with autograd through the oracle (same ReLU decisions, see the test above)."""
    import torch.nn.functional as F
    sd = synthetic_state_dict(2, 'random')
    x = synthetic_panoramas(2, seed=43)
    gen = torch.Generator().manual_seed(10)
    y_bon, y_cor = torch.rand(2, 2, 1024, generator=gen) - 0.5, torch.rand(2, 1, 1024, generator=gen)
    net = HorizonNet('resnet50', True)
    net.load_state_dict(sd, strict=True)
    net = net.to(DEV).train()
    blocks = net.feature_extractor.list_blocks()
    for i in range(2):
        for m in blocks[i]:
            m.eval()
            for p in m.parameters():
                p.requires_grad = False
    frozen_bn = [n for n, m in net.named_modules() if isinstance(m, torch.nn.BatchNorm2d) and not m.training]
    assert len(frozen_bn) == 11
    bon, cor = net(x.to(DEV))
    loss = F.l1_loss(bon, y_bon.to(DEV)) + F.binary_cross_entropy_with_logits(cor, y_cor.to(DEV))
    loss.backward()
    net.check()
    masks = [t.cpu() for t in net.dropout_masks(net.last_dropout_seed, 2, DEV)]
    relu_masks = {}
    for i in range(69):
        name, y = net.debug_train_unit(i, 0)
        if not name.endswith('downsample.1'):
            relu_masks[name] = (y > 0).cpu()
    live = [k for k, p in net.named_parameters() if p.requires_grad]
    psd = {k: (v.clone().requires_grad_() if k in live else v) for k, v in sd.items()}
    tm = horizonnet_ref.TrainMode(masks=masks, frozen=frozen_bn, relu_masks=relu_masks)
    rbon, rcor = horizonnet_ref.forward(psd, x, train=tm)
    rloss = F.l1_loss(rbon, y_bon) + F.binary_cross_entropy_with_logits(rcor, y_cor)
    assert abs(loss.item() - rloss.item()) < 1e-5
    ref = dict(zip(live, torch.autograd.grad(rloss, [psd[k] for k in live])))
    gmax = max(float(v.abs().max()) for v in ref.values())
    worst = []
    for k, p in net.named_parameters():
        if k not in ref:
            assert p.grad is None, k
            continue
        worst.append((float((p.grad.cpu() - ref[k]).abs().max()) / (float(ref[k].abs().max()) + 1e-4 * gmax), k))
    worst.sort(reverse=True)
    assert worst[0][0] < 5e-3, worst[:8]
    after = net.state_dict()
    for n in frozen_bn:
        assert torch.equal(after[n + '.running_mean'].cpu(), sd[n + '.running_mean'])
        assert int(after[n + '.num_batches_tracked']) == 0


def test_training_loop_like_train_py_reduces_the_loss():
    """train.py:216-223 (Adam) + :272-281 (zero_grad / backward / step) on one fixed synthetic batch: the loss goes
    down, every optimizer step is seen by the library (weights re-uploaded), and eval mode afterwards uses the moved
    running statistics."""
    import torch.nn.functional as F
    sd = synthetic_state_dict(3, 'random')
    x = synthetic_panoramas(2, seed=47).to(DEV)
    gen = torch.Generator().manual_seed(12)
    y_bon = (torch.rand(2, 2, 1024, generator=gen) - 0.5).to(DEV)
    y_cor = torch.rand(2, 1, 1024, generator=gen).to(DEV)
    net = _train_net(sd, True)
    opt = torch.optim.Adam(net.parameters(), lr=1e-3, betas=(0.9, 0.999))
    losses = []
    for _ in range(5):
        torch.manual_seed(0)                    # the same dropout masks every step: the loss curve is not noise
        opt.zero_grad()
        bon, cor = net(x)
        loss = F.l1_loss(bon, y_bon) + F.binary_cross_entropy_with_logits(cor, y_cor)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    net.check()
    assert losses[-1] < losses[0] - 0.02, losses
    assert all(np.isfinite(losses))
    net.eval()
    with torch.no_grad():
        ebon, ecor = net(x)
        rbon, rcor = horizonnet_ref.forward({k: v.cpu() for k, v in net.state_dict().items()}, x.cpu())
    assert (ebon.cpu() - rbon).abs().max().item() < 2e-4 and (ecor.cpu() - rcor).abs().max().item() < 2e-4


def test_training_batch_growth_on_one_library_handle():
    """The tape buffers are laid out for the first training batch; a larger one later on the same handle (created by an
    eval forward of the larger batch) frees and re-lays them out.  The larger step must equal a fresh model's step."""
    import torch.nn.functional as F
    sd = synthetic_state_dict(4, 'random')
    x = synthetic_panoramas(2, seed=51).to(DEV)
    y_bon, y_cor = torch.zeros(2, 2, 1024, device=DEV), torch.full((2, 1, 1024), 0.5, device=DEV)

    def step(net, xb):
        torch.manual_seed(3)
        net.zero_grad()
        bon, cor = net(xb)
        n = xb.shape[0]
        loss = F.l1_loss(bon, y_bon[:n]) + F.binary_cross_entropy_with_logits(cor, y_cor[:n])
        loss.backward()
        return loss.item(), net.linear.weight.grad.clone(), net.feature_extractor.encoder.conv1[1].weight.grad.clone()

    net = _train_net(sd, True)
    net.eval()
    with torch.no_grad():
        net(x)                                   # handle with max_batch = 2
    net.train()
    step(net, x[:1])                             # tape laid out for batch 1 ...
    net.load_state_dict(sd)                      # (undo the running-statistics update of that step)
    l2, g2a, g2b = step(net, x)                  # ... and again for batch 2
    fresh = _train_net(sd, True)
    l2f, g2fa, g2fb = step(fresh, x)
    net.check()
    assert abs(l2 - l2f) < 1e-6
    # (the weight gradients are fp32 atomic sums: equal up to summation order)
    for a, b in ((g2a, g2fa), (g2b, g2fb)):
        assert float((a - b).abs().max()) <= 1e-4 * float(b.abs().max())
