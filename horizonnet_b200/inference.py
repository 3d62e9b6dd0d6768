"""Device-side inference around the forward (reference inference.py).

``tta_forward(net, x, flip, rotate)`` replaces the first half of the reference's ``inference()`` (inference.py:32-62,
77-93): ``augment`` (numpy flip / roll on the host), ``net(x.to(device))``, two ``.cpu()`` round trips, ``sigmoid``,
``augment_undo(...).mean(0)`` and the boundary -> pixel-row conversion with clipping.  Here one panorama is uploaded
once; the views, the forward and the merge all run on the device.

The room-layout post-processing that follows (inference.py:95-139: floor/ceiling plane, wall-wall peaks, wall fitting,
the validity check with its cuboid fallback, corner assembly) runs on the device too (csrc/layout.cu):
  * ``infer_layout(net, x, ...)``: a batch of panoramas -> one (cor_id, z0, z1) per panorama;
  * ``layout_from_signals(y_bon_pix, y_cor, ...)``: the same post-processing on signals already on the device;
  * ``inference(net, x, device, ...)``: drop-in for the reference's ``inference()``;
  * ``python -m horizonnet_b200.inference --pth ... --img_glob ... --output_dir ...``: the reference's CLI, batched.
"""
import argparse
import ctypes
import glob
import json
import os
import sys

import numpy as np
import torch

from . import _lib
from ._spec import PANO_H, PANO_W

MODE_GENERAL, MODE_CUBOID, MODE_RAW = 0, 1, 2
STATUS_OK, STATUS_ASSERT, STATUS_RING = 0, 1, 2
MAX_WALLS, MAX_COR = 2048, 4096                # HN_LAYOUT_MAX_WALLS / HN_LAYOUT_MAX_COR
FALLBACK_MSG = 'Fail to generate valid general layout!! Generate cuboid as fallback.'   # inference.py:121-124

_workspaces = {}


def tta_forward(net, x, flip=False, rotate=()):
    """x: [1, 3, 512, 1024] float tensor (any device).  Returns (y_bon_ [2,1024] pixel rows, y_cor_ [1024]) as
    float32 numpy arrays -- the values the reference holds after inference.py:93 (before post-processing)."""
    if x.dim() != 4 or x.shape[0] != 1 or x.shape[1] != 3:
        raise ValueError('tta_forward expects one 3-channel panorama [1, 3, 512, 1024] (inference.py:196-200)')
    if x.shape[2] != PANO_H or x.shape[3] != PANO_W:
        raise NotImplementedError()
    dev = next(net.parameters()).device
    if dev.type != 'cuda':
        raise RuntimeError('horizonnet_b200 has no CPU path: move the model to a cuda device')
    shifts = [int(round(p * PANO_W)) for p in rotate]              # inference.py:40
    views = 1 + (1 if flip else 0) + len(shifts)
    h = net._handle(dev, max(views, 1))
    xd = x.detach().to(device=dev, dtype=torch.float32).contiguous()
    y_bon = torch.empty(2, PANO_W, device=dev, dtype=torch.float32)
    y_cor = torch.empty(PANO_W, device=dev, dtype=torch.float32)
    arr = (ctypes.c_int * max(len(shifts), 1))(*shifts) if shifts else None
    stream = torch.cuda.current_stream(dev).cuda_stream
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().hn_model_infer_tta(h['ptr'], xd.data_ptr(), 3, 1 if flip else 0, arr, len(shifts),
                                                 y_bon.data_ptr(), y_cor.data_ptr(), stream), 'hn_model_infer_tta')
    return y_bon.cpu().numpy(), y_cor.cpu().numpy()


# ------------------------------------------------------------------------------------------ layout
def _layout_args(force_cuboid, force_raw, min_v, r):
    """mode, float32 min_v and the peak window in pixels, as inference.py:99-109 derives them."""
    if force_raw:
        return MODE_RAW, 0.0, 1
    if min_v is None:
        min_v = 0 if force_cuboid else 0.05
    r_px = int(round(PANO_W * r / 2))
    if r_px < 1:
        raise ValueError('r must give a peak window of at least one column (int(round(1024 * r / 2)) >= 1)')
    return (MODE_CUBOID if force_cuboid else MODE_GENERAL), float(np.float32(min_v)), r_px


def _workspace(dev, B):
    """Device workspace of hn_layout, grown on demand and reused across calls."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    need = int(_lib.lib().hn_layout_workspace_bytes(B))
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.empty(need, dtype=torch.uint8, device=dev)
        _workspaces[key] = ws
    return ws


def _outputs(dev, B):
    return dict(cor_id=torch.empty(B, MAX_COR, 2, device=dev, dtype=torch.float32),
                n_cor=torch.empty(B, device=dev, dtype=torch.int32),
                z1=torch.empty(B, device=dev, dtype=torch.float32),
                status=torch.empty(B, 4, device=dev, dtype=torch.int32),
                peaks=torch.empty(B, PANO_W, device=dev, dtype=torch.int32),
                types=torch.empty(B, MAX_WALLS, device=dev, dtype=torch.int32))


def _ptrs(o):
    return [o[k].data_ptr() for k in ('cor_id', 'n_cor', 'z1', 'status', 'peaks', 'types')]


def layout_device(y_bon_pix, y_cor, force_cuboid=False, force_raw=False, min_v=None, r=0.05):
    """hn_layout on device signals y_bon_pix [B, 2, 1024] (pixel rows) and y_cor [B, 1024]; returns the raw device
    outputs (dict of tensors: cor_id [B, 4096, 2], n_cor, z1, status [B, 4], peaks, types)."""
    if y_bon_pix.dim() == 2:
        y_bon_pix, y_cor = y_bon_pix[None], y_cor.reshape(1, -1)
    y_cor = y_cor.reshape(y_cor.shape[0], -1)
    if y_bon_pix.shape[1:] != (2, PANO_W) or y_cor.shape != (y_bon_pix.shape[0], PANO_W):
        raise ValueError('layout expects y_bon_pix [B, 2, 1024] and y_cor [B, 1024]')
    dev = y_bon_pix.device
    if dev.type != 'cuda' or y_cor.device != dev:
        raise RuntimeError('horizonnet_b200 has no CPU path: the signals must be on one cuda device')
    mode, mv, r_px = _layout_args(force_cuboid, force_raw, min_v, r)
    B = y_bon_pix.shape[0]
    yb = y_bon_pix.detach().to(torch.float32).contiguous()
    yc = y_cor.detach().to(torch.float32).contiguous()
    out = _outputs(dev, B)
    stream = torch.cuda.current_stream(dev).cuda_stream
    with torch.cuda.device(dev):
        ws = _workspace(dev, B)
        _lib.check(_lib.lib().hn_layout(yb.data_ptr(), yc.data_ptr(), B, mode, mv, r_px, ws.data_ptr(), *_ptrs(out),
                                        stream), 'hn_layout')
    return out


def _results(out):
    """Device outputs -> [(cor_id [2K, 2] float32, z0, z1)], with the reference's fallback message and exceptions."""
    status = out['status'].cpu().numpy()
    n_cor = out['n_cor'].cpu().numpy()
    z1 = out['z1'].cpu().numpy()
    nmax = int(n_cor.max()) if len(n_cor) else 0
    cor_id = out['cor_id'][:, :nmax].cpu().numpy()
    for i in np.nonzero(status[:, 1])[0]:
        print(FALLBACK_MSG, file=sys.stderr)
    bad_assert = [int(i) for i in np.nonzero(status[:, 0] == STATUS_ASSERT)[0]]
    bad_ring = [int(i) for i in np.nonzero(status[:, 0] == STATUS_RING)[0]]
    if bad_assert or bad_ring:
        first = min(bad_assert + bad_ring)
        msg = 'layout post-processing failed as the reference does: AssertionError for panoramas %s, ' \
              'ValueError (wall ring shapely cannot build) for panoramas %s' % (bad_assert, bad_ring)
        raise (AssertionError if first in bad_assert else ValueError)(msg)
    return [(cor_id[i, :n_cor[i]].copy(), 50, np.float32(z1[i])) for i in range(len(n_cor))]


def layout_from_signals(y_bon_pix, y_cor, force_cuboid=False, force_raw=False, min_v=None, r=0.05):
    """inference.py:95-139 on the device for signals a caller already holds there (e.g. after its own
    ``forward_pipelined`` and decode): y_bon_pix [B, 2, 1024] boundary rows in pixels (inference.py:90-92),
    y_cor [B, 1024] sigmoid(cor).  Returns [(cor_id, z0, z1)] per panorama, like ``infer_layout``."""
    return _results(layout_device(y_bon_pix, y_cor, force_cuboid, force_raw, min_v, r))


def infer_layout_device(net, x, flip=False, rotate=(), force_cuboid=False, force_raw=False, min_v=None, r=0.05):
    """hn_model_infer_layout: batched TTA + forward + layout; returns (device outputs, y_bon_pix, y_cor)."""
    if x.dim() != 4 or x.shape[1] != 3:
        raise ValueError('infer_layout expects 3-channel panoramas [B, 3, 512, 1024] (inference.py:196-200)')
    if x.shape[2] != PANO_H or x.shape[3] != PANO_W:
        raise NotImplementedError()
    dev = next(net.parameters()).device
    if dev.type != 'cuda':
        raise RuntimeError('horizonnet_b200 has no CPU path: move the model to a cuda device')
    mode, mv, r_px = _layout_args(force_cuboid, force_raw, min_v, r)
    shifts = [int(round(p * PANO_W)) for p in rotate]              # inference.py:40
    views = 1 + (1 if flip else 0) + len(shifts)
    B = x.shape[0]
    h = net._handle(dev, max(1, min(B, 32 // views)) * views)   # up to 32 views per forward
    xd = x.detach().to(device=dev, dtype=torch.float32).contiguous()
    y_bon = torch.empty(B, 2, PANO_W, device=dev, dtype=torch.float32)
    y_cor = torch.empty(B, PANO_W, device=dev, dtype=torch.float32)
    out = _outputs(dev, B)
    arr = (ctypes.c_int * max(len(shifts), 1))(*shifts) if shifts else None
    stream = torch.cuda.current_stream(dev).cuda_stream
    with torch.cuda.device(dev):
        ws = _workspace(dev, B)
        _lib.check(_lib.lib().hn_model_infer_layout(h['ptr'], xd.data_ptr(), B, 1 if flip else 0, arr, len(shifts),
                                                    mode, mv, r_px, ws.data_ptr(), y_bon.data_ptr(), y_cor.data_ptr(),
                                                    *_ptrs(out), stream), 'hn_model_infer_layout')
    return out, y_bon, y_cor


def infer_layout(net, x, flip=False, rotate=(), force_cuboid=False, force_raw=False, min_v=None, r=0.05):
    """x: [B, 3, 512, 1024].  Returns one (cor_id [2K, 2] float32, z0, z1) per panorama: what the reference's
    ``inference()`` returns for each panorama alone.  Where the reference would raise for some panorama this raises
    the same exception type (AssertionError, or ValueError for a wall ring shapely cannot build) naming the indices;
    the reference's fallback message is printed once per panorama that fell back to the cuboid."""
    return _results(infer_layout_device(net, x, flip, rotate, force_cuboid, force_raw, min_v, r)[0])


def inference(net, x, device, flip=False, rotate=[], visualize=False, force_cuboid=False, force_raw=False,
              min_v=None, r=0.05):
    """Drop-in for the reference's inference() (inference.py:65-141): x [1, 3, 512, 1024]; returns
    (cor_id, z0, z1, vis_out) with vis_out None.  ``device`` is where ``net`` lives (a cuda device)."""
    if visualize:
        raise NotImplementedError('visualize draws on the host and is not part of horizonnet_b200')
    if x.dim() != 4 or x.shape[0] != 1:
        raise ValueError('inference expects one panorama [1, 3, 512, 1024]')
    cor_id, z0, z1 = infer_layout(net, x, flip, rotate, force_cuboid, force_raw, min_v, r)[0]
    return cor_id, z0, z1, None


# ------------------------------------------------------------------------------------------ CLI (inference.py:144-216)
def load_image(path):
    """inference.py:196-200: RGB(A) image -> [1, 3, 512, 1024] float32 in [0, 1] (BICUBIC resize if needed)."""
    from PIL import Image
    img_pil = Image.open(path)
    if img_pil.size != (1024, 512):
        img_pil = img_pil.resize((1024, 512), Image.BICUBIC)
    img_ori = np.array(img_pil)[..., :3].transpose([2, 0, 1]).copy()
    return torch.FloatTensor(np.array([img_ori / 255]))


def load_trained_model(path):
    """misc/utils.py load_trained_model with this package's HorizonNet."""
    from .model import HorizonNet
    state_dict = torch.load(path, map_location='cpu')
    net = HorizonNet(**state_dict['kwargs'])
    net.load_state_dict(state_dict['state_dict'])
    return net


def main(argv=None):
    parser = argparse.ArgumentParser(formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    parser.add_argument('--pth', required=True, help='path to load saved checkpoint.')
    parser.add_argument('--img_glob', required=True, help='quoted glob of aligned panoramas')
    parser.add_argument('--output_dir', required=True)
    parser.add_argument('--flip', action='store_true', help='left-right flip augmentation (x2 views)')
    parser.add_argument('--rotate', nargs='*', default=[], type=float,
                        help='horizontal rotations, fractions of the image width (one view each)')
    parser.add_argument('--r', default=0.05, type=float)
    parser.add_argument('--min_v', default=None, type=float)
    parser.add_argument('--force_cuboid', action='store_true')
    parser.add_argument('--force_raw', action='store_true')
    parser.add_argument('--batch', default=16, type=int, help='panoramas per device call')
    args = parser.parse_args(argv)

    paths = sorted(glob.glob(args.img_glob))
    if len(paths) == 0:
        print('no images found')
    for path in paths:
        assert os.path.isfile(path), '%s not found' % path
    if not os.path.isdir(args.output_dir):
        print('Output directory %s not existed. Create one.' % args.output_dir)
        os.makedirs(args.output_dir)
    net = load_trained_model(args.pth).to('cuda')
    net.eval()
    with torch.no_grad():
        for i in range(0, len(paths), max(args.batch, 1)):
            chunk = paths[i:i + max(args.batch, 1)]
            x = torch.cat([load_image(p) for p in chunk], 0)
            results = infer_layout(net, x, flip=args.flip, rotate=args.rotate, force_cuboid=args.force_cuboid,
                                   force_raw=args.force_raw, min_v=args.min_v, r=args.r)
            for path, (cor_id, z0, z1) in zip(chunk, results):
                k = os.path.split(path)[-1][:-4]
                with open(os.path.join(args.output_dir, k + '.json'), 'w') as f:
                    json.dump({'z0': float(z0), 'z1': float(z1), 'uv': [[float(u), float(v)] for u, v in cor_id]}, f)


if __name__ == '__main__':
    main()
