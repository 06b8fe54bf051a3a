"""Kernel-level parity against the REFERENCE'S OWN CUDA extension `localattention`, compiled unmodified for sm_100a by
oracle/build_ref.py: its outputs on the seeded inputs below are stored in tests/golden/locatt_ref.pt
(tools/ref_goldens.py), each compared at fixed, seeded positions.

  (i)   the five drop-in entry points of projects/.../locatt_ops (forward + the three backward mappings, served by
        di_locatt_{cc2k,ck2c_ori,ck2c_loc}_f32) == the reference functions (localAttention.cpp:61-73), incl. non-square
        maps and kH != kW;
  (ii)  the fused window kernels (FFMA, mma.sync 3xTF32 / bf16 split, tcgen05) == reference
        similar_forward -> softmax(./sqrt(C)) -> weighting_forward (encoder_utils.py:132-134);
  (iii) the CPU oracle's window ops == the reference kernels (this pins the one op whose committed golden had to use a
        stand-in, SURVEY.md Appendix B).
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_err
from tools import ref_goldens as rg
from tools.ref_goldens import sampled_rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dev():
    return torch.device('cuda:0')


@pytest.fixture(scope='module')
def gold():
    return torch.load(os.path.join(ROOT, 'tests', 'golden', 'locatt_ref.pt'), weights_only=True)


def _drop_in():
    from projects.mmdet3d_plugin.models.utils.ops.locatt_ops import localattention
    return localattention


@pytest.mark.parametrize('N,C,H,W,kH,kW', rg.DROP_IN_SHAPES)
def test_drop_in_entry_points_equal_reference_extension(gold, N, C, H, W, kH, kW):
    ours = _drop_in()
    inputs = [t.to(dev()) for t in rg.drop_in_inputs(N, C, H, W, kH, kW)]
    tol = 2e-6           # both sides accumulate in fp64 and round once; the summation order differs
    for name, (fn, args) in rg.drop_in_calls(*inputs, kH, kW).items():
        assert sampled_rel_err(getattr(ours, fn)(*args), gold['drop_in', (N, C, H, W, kH, kW), name]) < tol, name


def test_drop_in_backward_is_the_gradient_of_the_forward():
    """The backward mappings, used the way the reference's autograd Functions use them (encoder_utils.py:36-81),
    equal torch.autograd of the oracle's differentiable restatement."""
    import oracle.mmri as om
    ours = _drop_in()
    g = torch.Generator().manual_seed(7)
    N, C, H, W, k = 1, 8, 7, 9, 5
    q = torch.randn(N, C, H, W, generator=g, dtype=torch.float64, requires_grad=True)
    kk = torch.randn(N, C, H, W, generator=g, dtype=torch.float64, requires_grad=True)
    v = torch.randn(N, C, H, W, generator=g, dtype=torch.float64, requires_grad=True)
    w = F.softmax(om.window_similarity(q, kk, k) / np.sqrt(C), -1)
    out = om.window_weighting(v, w, k)
    go = torch.randn(out.shape, generator=g, dtype=torch.float64)
    gq, gk, gv = torch.autograd.grad(out, (q, kk, v), go)
    # the same chain through the drop-in kernels
    f = lambda t: t.detach().float().to(dev())
    sim = ours.similar_forward(f(q), f(kk), k, k)
    wd = F.softmax(sim / np.sqrt(C), -1)
    g_w = ours.weighting_backward_weight(f(v), f(go), k, k)            # d out / d weight
    g_v = ours.weighting_backward_ori(wd, f(go), k, k)                 # d out / d v
    g_sim = (wd * (g_w - (g_w * wd).sum(-1, keepdim=True))) / np.sqrt(C)
    g_q = ours.similar_backward(f(kk), g_sim, k, k, True)
    g_k = ours.similar_backward(f(q), g_sim, k, k, False)
    for name, a, b in (('dq', g_q, gq), ('dk', g_k, gk), ('dv', g_v, gv)):
        assert rel_err(a.cpu().double(), b) < 2e-5, name


@pytest.mark.parametrize('kernel', ['tcgen05', 'mma-bf16split', 'mma-3xtf32', 'ffma'])
@pytest.mark.parametrize('N,H,W', rg.FUSED_SHAPES)
def test_fused_window_equals_reference_similar_softmax_weighting(gold, kernel, N, H, W):
    from deepinteraction_b200 import ops, fold, _lib
    C, k = 128, 9
    q, kk, v = (t.to(dev()) for t in rg.fused_inputs(N, H, W, C))
    rows = lambda t: t.permute(0, 2, 3, 1).reshape(-1, C).contiguous()
    if kernel == 'tcgen05':
        out = ops.lcab_window_tc(fold.split_rows(rows(q), 3), fold.split_rows(rows(kk), 3), fold.split_rows(rows(v), 3),
                                 N, H, W, C)
    else:
        _lib.lib().di_set_window_ffma({'mma-bf16split': 0, 'ffma': 1, 'mma-3xtf32': 2}[kernel])
        try:
            out = ops.lcab_window(rows(q), rows(kk), rows(v), N, H, W, C, k)
        finally:
            _lib.lib().di_set_window_ffma(0)
    got = out.view(N, H, W, C).permute(0, 3, 1, 2)
    assert sampled_rel_err(got, gold['fused', (N, H, W)]) < 5e-5


def test_cpu_oracle_window_ops_equal_reference_kernels(gold):
    """Both weightings are applied to the softmax of the oracle's similarity."""
    import oracle.mmri as om
    q, kk, v, w, k = rg.oracle_window_inputs()
    assert sampled_rel_err(om.window_similarity(q, kk, k), gold['oracle', 'similar_forward']) < 2e-6
    assert sampled_rel_err(om.window_weighting(v, w, k), gold['oracle', 'weighting_forward']) < 2e-6
