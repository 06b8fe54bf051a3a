#!/usr/bin/env python
"""Goldens that pin the tests to the reference project without needing it at test time.

    python tools/ref_goldens.py configs --ref REFERENCE_TREE   # -> tests/golden/ref_configs.pt   (CPU)
    python tools/ref_goldens.py locatt [--out FILE]             # -> tests/golden/locatt_ref.pt   (B200)

`configs` executes the reference's two nuScenes config files (registry.load_config) and keeps what the plug-in
builds from them: `plugin`, `plugin_dir` and the detector's `type`, `imgpts_neck`, `pts_bbox_head`, `train_cfg` and
`test_cfg`.

`locatt` runs the reference's own CUDA extension `localattention` (compiled by oracle/build_ref.py into oracle/_ref/)
on the seeded inputs of the window-op parity tests (tests/test_gpu_locatt_ref.py, tests/test_gpu_backward.py).  Every
output is stored as its shape, max |value| and the values at SAMPLE fixed, seeded positions (all of them for smaller
outputs): `sampled_rel_err` is then the tests' max|a - b| / max|b| over those positions.  The inputs are not stored;
the case functions below re-create them from their seeds.
"""
import argparse
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
SAMPLE = 512
REF_CONFIGS = ('Fusion_0075_refactor', 'Fusion_0075_plusplus')
MODEL_KEYS = ('type', 'imgpts_neck', 'pts_bbox_head', 'train_cfg', 'test_cfg')

# (N, C, H, W, kH, kW): the five drop-in entry points of locatt_ops
DROP_IN_SHAPES = [(2, 16, 9, 13, 9, 9), (1, 128, 20, 17, 9, 9), (2, 8, 7, 11, 3, 5), (1, 32, 5, 6, 5, 3)]
# (N, H, W) at C = 128, k = 9: similar_forward -> softmax(. / sqrt(C)) -> weighting_forward, the fused window kernels
FUSED_SHAPES = [(2, 40, 33), (1, 17, 50)]
# (N, C, H, W, k): the pixel-major window kernels of the training step
BACKWARD_SHAPES = [(2, 128, 11, 14, 9), (1, 32, 7, 9, 9), (1, 256, 6, 5, 5)]


def ref_config(name):
    """The stored part of the reference config `name` (one of REF_CONFIGS)."""
    return torch.load(os.path.join(GOLDEN, 'ref_configs.pt'), weights_only=True)[name]


def drop_in_inputs(N, C, H, W, kH, kW):
    g = torch.Generator().manual_seed(100 + C)
    x_ori = torch.randn(N, C, H, W, generator=g)
    x_loc = torch.randn(N, C, H, W, generator=g)
    wgt = torch.randn(N, H, W, kH * kW, generator=g)
    grad_c = torch.randn(N, C, H, W, generator=g)
    return x_ori, x_loc, wgt, grad_c


def drop_in_calls(x_ori, x_loc, wgt, grad_c, kH, kW):
    """name -> (entry point, arguments); the same calls go to the reference extension and to the drop-in module."""
    return {'similar_forward': ('similar_forward', (x_ori, x_loc, kH, kW)),
            'similar_backward(is_ori)': ('similar_backward', (x_loc, wgt, kH, kW, True)),
            'similar_backward(is_loc)': ('similar_backward', (x_ori, wgt, kH, kW, False)),
            'weighting_forward': ('weighting_forward', (x_ori, wgt, kH, kW)),
            'weighting_backward_ori': ('weighting_backward_ori', (wgt, grad_c, kH, kW)),
            'weighting_backward_weight': ('weighting_backward_weight', (x_ori, grad_c, kH, kW))}


def fused_inputs(N, H, W, C=128):
    g = torch.Generator().manual_seed(31 + H)
    return tuple(torch.randn(N, C, H, W, generator=g) for _ in range(3))


def oracle_window_inputs():
    """q, k, v of the CPU-oracle check, and the softmax weights both sides' weighting is applied to."""
    import oracle.mmri as om
    g = torch.Generator().manual_seed(5)
    N, C, H, W, k = 2, 64, 11, 14, 9
    q, kk, v = (torch.randn(N, C, H, W, generator=g) for _ in range(3))
    w = F.softmax(om.window_similarity(q, kk, k) / np.sqrt(C), -1)
    return q, kk, v, w, k


def backward_inputs(N, C, H, W, ks):
    g = torch.Generator().manual_seed(7 + C)
    a = torch.randn(N, C, H, W, generator=g)
    b = torch.randn(N, C, H, W, generator=g)
    w = torch.randn(N, H, W, ks * ks, generator=g)
    return a, b, w


def backward_calls(a, b, w, ks):
    return {'similar_forward(a,b)': ('similar_forward', (a, b, ks, ks)),
            'weighting_forward(b,w)': ('weighting_forward', (b, w, ks, ks)),
            'similar_backward(b,w,is_ori)': ('similar_backward', (b, w, ks, ks, True)),
            'similar_backward(a,w,is_loc)': ('similar_backward', (a, w, ks, ks, False)),
            'weighting_backward_ori(w,a)': ('weighting_backward_ori', (w, a, ks, ks)),
            'weighting_backward_weight(b,a)': ('weighting_backward_weight', (b, a, ks, ks))}


def sample_index(n):
    if n <= SAMPLE:
        return torch.arange(n)
    return torch.randperm(n, generator=torch.Generator().manual_seed(0))[:SAMPLE].sort().values


def entry(t):
    t = t.detach().float().cpu()
    return dict(shape=tuple(t.shape), absmax=float(t.abs().max()), vals=t.reshape(-1)[sample_index(t.numel())])


def sampled_rel_err(got, gold):
    """max|got - ref| / max|ref| over the stored positions of the reference output `gold`."""
    assert tuple(got.shape) == gold['shape'], (tuple(got.shape), gold['shape'])
    got = got.detach().float().cpu().reshape(-1)[sample_index(got.numel())]
    return float((got - gold['vals']).abs().max() / max(gold['absmax'], 1e-12))


def make_configs(ref):
    from projects.mmdet3d_plugin.registry import load_config
    out = {}
    for name in REF_CONFIGS:
        cfg = load_config(os.path.join(ref, 'projects', 'configs', 'nuscenes', name + '.py'))
        out[name] = dict(plugin=cfg['plugin'], plugin_dir=cfg['plugin_dir'],
                         model={k: cfg['model'][k] for k in MODEL_KEYS if k in cfg['model']})
    return out


def make_locatt():
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import build_ref
    ref = build_ref.load()
    assert ref is not None, 'oracle/_ref/localattention.so not built (python oracle/build_ref.py)'
    dev = torch.device('cuda:0')
    run = lambda fn, args: getattr(ref, fn)(*[a.to(dev) if torch.is_tensor(a) else a for a in args])
    out = dict(sample=SAMPLE)
    for shp in DROP_IN_SHAPES:
        for name, (fn, args) in drop_in_calls(*drop_in_inputs(*shp), *shp[4:]).items():
            out['drop_in', shp, name] = entry(run(fn, args))
    for N, H, W in FUSED_SHAPES:
        C, k = 128, 9
        q, kk, v = (t.to(dev) for t in fused_inputs(N, H, W, C))
        out['fused', (N, H, W)] = entry(ref.weighting_forward(v, F.softmax(ref.similar_forward(q, kk, k, k) / np.sqrt(C), -1), k, k))
    q, kk, v, w, k = oracle_window_inputs()
    out['oracle', 'similar_forward'] = entry(run('similar_forward', (q, kk, k, k)))
    out['oracle', 'weighting_forward'] = entry(run('weighting_forward', (v, w, k, k)))
    for shp in BACKWARD_SHAPES:
        for name, (fn, args) in backward_calls(*backward_inputs(*shp), shp[4]).items():
            out['backward', shp, name] = entry(run(fn, args))
    torch.cuda.synchronize()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('what', choices=['configs', 'locatt'])
    ap.add_argument('--ref', help='configs: root of the reference tree')
    ap.add_argument('--out', help='default: tests/golden/ref_configs.pt or tests/golden/locatt_ref.pt')
    args = ap.parse_args()
    if args.what == 'configs':
        assert args.ref, '--ref is required'
        obj, out = make_configs(args.ref), args.out or os.path.join(GOLDEN, 'ref_configs.pt')
    else:
        obj, out = make_locatt(), args.out or os.path.join(GOLDEN, 'locatt_ref.pt')
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    torch.save(obj, out)
    print(out, '%.0f KiB' % (os.path.getsize(out) / 1024))


if __name__ == '__main__':
    main()
