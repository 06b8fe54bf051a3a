"""Training side on the GPU (deepinteraction_b200/{backward,train}.py + csrc/{lcab_bwd,bn_train}.cu, the I2P kernels of
geometry.cu): window kernels against the reference's own CUDA extension (its outputs stored in tests/golden/locatt_ref.pt)
and the CPU oracle's autograd; input / parameter gradients of the attention blocks and of the whole encoder against
autograd through the oracle with BatchNorm in eval mode (folded weights) and in training mode (batch statistics; the
oracle's .train() behaviour is itself pinned to the reference by tests/golden/{lcab,encoder}_train.pt); the I2P attention dropout with the product's mask injected into the oracle."""
import os

import pytest
import torch

from conftest import rel_err
from tools.ref_goldens import BACKWARD_SHAPES, backward_inputs, sampled_rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dev():
    return torch.device('cuda:0')


def rows(t):           # (N, C, H, W) -> [N*H*W, C]
    return t.permute(0, 2, 3, 1).reshape(-1, t.shape[1]).contiguous()


@pytest.mark.parametrize('N,C,H,W,ks', BACKWARD_SHAPES)
def test_window_backward_kernels_match_reference_extension(N, C, H, W, ks):
    """di_win_dot / gather / scatter (pixel-major) == the reference localattention functions (NCHW) they stand for."""
    from deepinteraction_b200 import ops
    gold = torch.load(os.path.join(ROOT, 'tests', 'golden', 'locatt_ref.pt'), weights_only=True)
    ref = lambda name: gold['backward', (N, C, H, W, ks), name]
    a, b, w = (t.to(dev()) for t in backward_inputs(N, C, H, W, ks))
    ar, br, wr = rows(a), rows(b), w.reshape(-1, ks * ks).contiguous()
    back = lambda r: r.view(N, H, W, C).permute(0, 3, 1, 2)
    tol = 3e-6
    assert sampled_rel_err(ops.win_dot(ar, br, N, H, W, ks).view(N, H, W, -1), ref('similar_forward(a,b)')) < tol
    assert sampled_rel_err(back(ops.win_gather(wr, br, N, H, W, ks)), ref('weighting_forward(b,w)')) < tol
    assert sampled_rel_err(back(ops.win_gather(wr, br, N, H, W, ks)), ref('similar_backward(b,w,is_ori)')) < tol
    assert sampled_rel_err(back(ops.win_scatter(wr, ar, N, H, W, ks)), ref('similar_backward(a,w,is_loc)')) < tol
    assert sampled_rel_err(back(ops.win_scatter(wr, ar, N, H, W, ks)), ref('weighting_backward_ori(w,a)')) < tol
    assert sampled_rel_err(ops.win_dot(ar, br, N, H, W, ks).view(N, H, W, -1), ref('weighting_backward_weight(b,a)')) < tol


def test_softmax_relu_colsum_kernels():
    from deepinteraction_b200 import ops
    g = torch.Generator().manual_seed(3)
    S = torch.randn(500, 81, generator=g) * 3
    dA = torch.randn(500, 81, generator=g)
    Sg = S.clone().requires_grad_(True)
    A_ref = torch.softmax(Sg * 0.37, -1)
    (A_ref * dA).sum().backward()
    A = ops.win_softmax(S.to(dev()), 0.37)
    assert rel_err(A.cpu(), A_ref.detach()) < 2e-6
    assert rel_err(ops.win_softmax_bwd(A, dA.to(dev()), 0.37).cpu(), Sg.grad) < 5e-6
    y, dy = torch.randn(1001, 36, generator=g), torch.randn(1001, 36, generator=g)
    assert torch.equal(ops.relu_bwd(dy.to(dev()), y.to(dev())).cpu(), dy * (y > 0))
    x = torch.randn(70001, 128, generator=g)
    assert rel_err(ops.col_sum(x.to(dev())).cpu(), x.double().sum(0).float()) < 2e-6


@pytest.mark.parametrize('self_attn', [True, False])
def test_lcab_backward_matches_oracle_autograd(self_attn):
    """d target / d source / d folded weights and biases of the five Conv+BN layers vs torch autograd through the CPU oracle
    block in eval mode; the folded-weight gradient maps to the convolution weight by the BN scale."""
    import oracle.mmri as om
    from deepinteraction_b200 import mmri, synth, backward
    torch.manual_seed(31)
    C, N, H, W = 128, 2, 12, 20
    blk = om.LocalContextAttentionBlock(C, C, 9).eval()
    synth.randomize_norm_stats(blk, 31)
    g = torch.Generator().manual_seed(31)
    xt = torch.randn(N, C, H, W, generator=g).requires_grad_(True)
    xs = xt if self_attn else torch.randn(N, C, H, W, generator=g).requires_grad_(True)
    G = torch.randn(N, C, H, W, generator=g)
    with torch.enable_grad():
        out = blk(xt, xs)
        (out * G).sum().backward()
    pk = mmri._pack_lcab(blk, dev())
    t = rows(xt.detach()).to(dev())
    s = t if self_attn else rows(xs.detach()).to(dev())
    r = backward.lcab_backward(pk, t, s, N, H, W, rows(G).to(dev()))
    tol = 2e-4          # bf16-split tensor-core products (1e-5 each) through a five-layer chain
    assert rel_err(r['d_target'].cpu(), rows(xt.grad)) < tol
    if self_attn:
        assert r['d_source'] is None
    else:
        assert rel_err(r['d_source'].cpu(), rows(xs.grad)) < tol
    layers = dict(q1=blk.query_project[0], q2=blk.query_project[1], k1=blk.key_project[0], k2=blk.key_project[1],
                  v=blk.value_project)
    for name, m in layers.items():
        dW, db = r[name]
        scale = (m.bn.weight / torch.sqrt(m.bn.running_var + m.bn.eps)).detach()
        want_w = m.conv.weight.grad[:, :, 0, 0]                         # = dW_folded * scale (rows)
        assert rel_err(dW.cpu() * scale[:, None], want_w) < tol, name
        assert rel_err(db.cpu(), m.bn.bias.grad) < tol, name
    # autograd wrapper: same input gradients through torch.autograd
    tt = t.clone().requires_grad_(True)
    ss = tt if self_attn else s.clone().requires_grad_(True)
    with torch.enable_grad():
        o = backward.LCABFunction.apply(pk, tt, ss, N, H, W)
        assert rel_err(o.detach().cpu(), rows(out.detach())) < 2e-4
        (o * rows(G).to(dev())).sum().backward()
    assert rel_err(tt.grad.cpu(), rows(xt.grad)) < tol


@pytest.mark.parametrize('aug', [False, True])
def test_i2p_backward_matches_oracle_autograd(aug):
    """MMRI_I2P (BASELINE config 1 shapes: 32x32 BEV, C = 64, one 64x64 camera map, batch 2): gradients w.r.t. the BEV map, the
    image map and the attention module's own parameters vs torch autograd through the CPU oracle."""
    import oracle.mmri as om
    from deepinteraction_b200 import mmri, synth, fold, geom, backward
    from test_gpu_encoder import _cfg1_frame
    seed = 1100
    torch.manual_seed(seed)
    m = om.MMRI_I2P(64, 64, 0.1).eval()
    synth.randomize_norm_stats(m, seed)
    fr = _cfg1_frame(seed, aug)
    g = torch.Generator().manual_seed(seed)
    pts = fr['pts_feats'].clone().requires_grad_(True)                  # (B, C, Y, X)
    img = fr['img_feats'].clone().requires_grad_(True)                  # (B*V, C, h, w), V = 1
    B = pts.shape[0]
    G = torch.randn(pts.shape, generator=g)
    with torch.enable_grad():
        out = m(pts, img.view(B, 1, *img.shape[1:]), fr['img_metas'], fr['pts_metas'])
        (out * G).sum().backward()
    d = dev()
    mha = m.learnedAlign
    M1, c1, M2, c2 = fold.i2p_fold(mha)
    pack = (fold.Weight(M1, d), fold.dev(c1, d), fold.Weight(M2, d), fold.dev(c2, d))
    enc = mmri.DeepInteractionEncoder(1, 64, 64, 64)
    pm = enc._canon_pts_metas(fr['pts_metas'], d)
    proj, _ = geom.camera_rows(fr['img_metas'], d)
    nhwc = lambda t: t.detach().permute(0, 2, 3, 1).contiguous().to(d)
    r = backward.i2p_backward(pack, nhwc(pts), nhwc(img), pm, proj, 1, (256, 256), nhwc(G))
    tol = 1e-4
    assert rel_err(r['d_pts'].permute(0, 3, 1, 2).cpu(), pts.grad) < tol
    assert rel_err(r['d_img'].permute(0, 3, 1, 2).cpu(), img.grad) < tol
    assert float(pts.grad.abs().max()) > 0 and float(img.grad.abs().max()) > 0
    pg = fold.i2p_unfold_grads(mha, r['dM1'], r['dc1'], r['dM2'], r['dc2'])
    Wq_g, Wk_g, Wv_g = (mha.in_proj_weight.grad.chunk(3, 0) if mha._qkv_same_embed_dim else
                        (mha.q_proj_weight.grad, mha.k_proj_weight.grad, mha.v_proj_weight.grad))
    bq_g, bk_g, bv_g = mha.in_proj_bias.grad.chunk(3, 0)
    for name, want in (('Wq', Wq_g), ('Wk', Wk_g), ('Wv', Wv_g), ('bq', bq_g), ('bv', bv_g),
                       ('Wo', mha.out_proj.weight.grad), ('bo', mha.out_proj.bias.grad)):
        assert rel_err(pg[name].float(), want) < tol, name
    assert float(bk_g.abs().max()) < 1e-4 * float(bq_g.abs().max() + 1e-12)          # the key bias has no influence


def test_encoder_backward_matches_oracle_autograd():
    """Whole base encoder (2 layers: I2P, BEVWarp sampling + P2I, both self-attention blocks, fuse convolutions, 3x3 shared
    convolutions) with BatchNorm in eval mode: gradients of a random linear functional of the three outputs w.r.t. the two input
    feature maps, and a few folded parameter gradients, vs torch autograd through the CPU oracle."""
    import oracle.mmri as om
    from deepinteraction_b200 import mmri, synth, backward
    from tools.make_goldens import small_frame
    seed = 1560
    torch.manual_seed(seed)
    m = om.DeepInteractionEncoder(2, 64, 64, 128).eval()
    synth.randomize_norm_stats(m, seed)
    fr = small_frame(seed, aug=True, views=2, c_img=64, c_pts=64, bev=36, batch=1)
    g = torch.Generator().manual_seed(seed)
    xi = fr['img_feats'].clone().requires_grad_(True)
    xp = fr['pts_feats'].clone().requires_grad_(True)
    with torch.enable_grad():
        o_img, (o_pc, o_p) = m(xi, xp, fr['img_metas'], fr['pts_metas'])
        G_img, G_pc, G_p = (torch.randn(t.shape, generator=g) for t in (o_img, o_pc, o_p))
        ((o_img * G_img).sum() + (o_pc * G_pc).sum() + (o_p * G_p).sum()).backward()
    enc = mmri.DeepInteractionEncoder(2, 64, 64, 128)
    enc.load_state_dict(m.state_dict(), strict=True)
    enc = enc.to(dev()).eval()
    d = dev()
    nhwc = lambda t: t.detach().permute(0, 2, 3, 1).contiguous().to(d)
    pm = {k: (v.to(d) if torch.is_tensor(v) else [p.to(d) for p in v]) for k, v in fr['pts_metas'].items()}
    r = backward.encoder_backward(enc, fr['img_feats'].to(d), fr['pts_feats'].to(d), fr['img_metas'], pm, nhwc(G_img), nhwc(G_pc),
                                  nhwc(G_p))
    tol = 1e-3          # the forward intermediates carry the inference path's bf16-split rounding (1e-5 per layer)
    e_i = rel_err(r['d_img_feats'].permute(0, 3, 1, 2).cpu(), xi.grad)
    e_p = rel_err(r['d_pts_feats'].permute(0, 3, 1, 2).cpu(), xp.grad)
    print('encoder backward: d img_feats %.2e, d pts_feats %.2e' % (e_i, e_p))
    assert e_i < tol and e_p < tol
    # parameter gradients of the last layer: value_project of I_IML (conv weight via the BN scale) and the I2P output bias
    blk = m.fusion_blocks[1]
    vp = blk.I_IML.value_project
    scale = (vp.bn.weight / torch.sqrt(vp.bn.running_var + vp.bn.eps)).detach()
    dW, db = r['layers'][1]['i_iml']['v']
    assert rel_err(dW.cpu() * scale[:, None], vp.conv.weight.grad[:, :, 0, 0]) < tol
    assert rel_err(db.cpu(), vp.bn.bias.grad) < tol
    assert rel_err(r['layers'][1]['i2p'][3].cpu(), blk.I2P_block.learnedAlign.out_proj.bias.grad) < tol
    # the two 3x3 shared convolutions (weights and biases)
    for name, conv in (('img', m.shared_conv_img), ('pts', m.shared_conv_pts)):
        dW, db = r['shared_conv'][name]
        assert rel_err(dW.cpu(), conv.weight.grad) < tol, name
        assert rel_err(db.cpu(), conv.bias.grad) < tol, name


def test_bn_train_kernels_match_torch():
    """di_bn_stats / di_bn_apply / di_bn_bwd against torch.nn.functional.batch_norm in training mode (+ReLU) and its autograd;
    a column with a large mean relative to its spread checks the two-pass moments."""
    import torch.nn.functional as F
    from deepinteraction_b200 import ops
    g = torch.Generator().manual_seed(3)
    for M, C, relu, affine in ((1000, 128, True, True), (37, 32, False, True), (5000, 64, True, False)):
        y = torch.randn(M, C, generator=g) * (torch.rand(C, generator=g) + 0.2) + torch.randn(C, generator=g) * 3
        y[:, 0] += 100.0
        gamma = (torch.rand(C, generator=g) + 0.5) if affine else None
        beta = torch.randn(C, generator=g) * 0.1 if affine else None
        rm, rv = torch.randn(C, generator=g) * 0.1, torch.rand(C, generator=g) + 0.5
        dz = torch.randn(M, C, generator=g)
        yr = y.double().clone().requires_grad_(True)
        gr = gamma.double().clone().requires_grad_(True) if affine else None
        br = beta.double().clone().requires_grad_(True) if affine else None
        rm_r, rv_r = rm.double().clone(), rv.double().clone()
        z_ref = F.batch_norm(yr, rm_r, rv_r, gr, br, True, 0.1, 1e-5)
        if relu:
            z_ref = F.relu(z_ref)
        (z_ref * dz.double()).sum().backward()
        d = dev()
        yd, rmd, rvd = y.to(d), rm.to(d), rv.to(d)
        gd, bd = (gamma.to(d), beta.to(d)) if affine else (None, None)
        mean, var = ops.bn_stats(yd, rmd, rvd, 0.1)
        z = ops.bn_apply(yd, mean, var, gd, bd, 1e-5, relu)
        dy, dg, db = ops.bn_bwd(dz.to(d), z if relu else None, yd, mean, var, gd, 1e-5)
        assert rel_err(z.cpu(), z_ref.detach().float()) < 2e-5, (M, C)
        assert rel_err(rmd.cpu(), rm_r.float()) < 1e-6 and rel_err(rvd.cpu(), rv_r.float()) < 1e-5
        assert rel_err(dy.cpu(), yr.grad.float()) < 5e-5, (M, C)
        if affine:
            assert rel_err(dg.cpu(), gr.grad.float()) < 2e-5 and rel_err(db.cpu(), br.grad.float()) < 2e-5


def _oracle_train_step(seed, dtype):
    import oracle.mmri as om
    from deepinteraction_b200 import synth
    from tools.make_goldens import small_frame
    torch.manual_seed(seed)
    m = om.DeepInteractionEncoder(2, 64, 64, 128)
    synth.randomize_norm_stats(m, seed)
    m.train()
    for blk in m.fusion_blocks:
        blk.I2P_block.learnedAlign.dropout = 0.0
    state0 = {k: v.clone() for k, v in m.state_dict().items()}
    m = m.to(dtype)
    fr = small_frame(seed, aug=True, views=2, c_img=64, c_pts=64, bev=36, batch=1)
    g = torch.Generator().manual_seed(seed)
    xi = fr['img_feats'].to(dtype).requires_grad_(True)
    xp = fr['pts_feats'].to(dtype).requires_grad_(True)
    pm = dict(fr['pts_metas'])
    pm['pillars'], pm['pts'] = pm['pillars'].to(dtype), [p.to(dtype) for p in pm['pts']]
    with torch.enable_grad():
        o_img, (o_pc, o_p) = m(xi, xp, fr['img_metas'], pm)
        Gs = [torch.randn(t.shape, generator=g) for t in (o_img, o_pc, o_p)]
        sum((o * G.to(dtype)).sum() for o, G in zip((o_img, o_pc, o_p), Gs)).backward()
    return dict(m=m, state0=state0, fr=fr, Gs=Gs, outs=[o.detach() for o in (o_img, o_pc, o_p)], d_in=(xi.grad, xp.grad),
                grads={n: p.grad for n, p in m.named_parameters()})


@pytest.mark.parametrize('self_attn', [True, False])
def test_lcab_train_mode_matches_oracle_autograd(self_attn):
    """LocalContextAttentionBlock with BatchNorm in TRAINING mode (train.LCABTrain): output, input gradients and every
    parameter gradient vs float64 autograd through the oracle block; bar per tensor = 1e-4 or 5x the error fp32 autograd
    makes on it (the batch-mean differences cancel heavily)."""
    import oracle.mmri as om
    from deepinteraction_b200 import mmri, synth, train, backward
    N, C, H, W = 2, 128, 11, 14
    torch.manual_seed(21)
    ref = om.LocalContextAttentionBlock(C, C, 9)
    synth.randomize_norm_stats(ref, 21)
    ref.train()
    state0 = {k: v.clone() for k, v in ref.state_dict().items()}
    g = torch.Generator().manual_seed(22)
    xt, xs, G = (torch.randn(N, C, H, W, generator=g) for _ in range(3))
    xs[:, :, :3] = 0.0                                  # rows of exact zeros, as the masked BEV warp produces

    def autograd(dtype):
        m = om.LocalContextAttentionBlock(C, C, 9)
        m.load_state_dict(state0)
        m = m.train().to(dtype)
        a = xt.to(dtype).requires_grad_(True)
        b = a if self_attn else xs.to(dtype).requires_grad_(True)
        with torch.enable_grad():
            o = m(a, b)
            (o * G.to(dtype)).sum().backward()
        return dict(out=o.detach(), d_t=a.grad, d_s=None if self_attn else b.grad, grads={n: p.grad for n, p in m.named_parameters()},
                    state=m.state_dict())
    r64, r32 = autograd(torch.float64), autograd(torch.float32)
    blk = mmri.LocalContextAttentionBlock(C, C, 9)
    blk.load_state_dict(state0, strict=True)
    blk = blk.to(dev()).train()
    t = rows(xt).to(dev())
    s_ = t if self_attn else rows(xs).to(dev())
    lt = train.LCABTrain(blk)
    grads = {}
    with backward._precise(), torch.no_grad():
        out = lt.forward(t, s_, N, H, W)
        d_t, d_s = lt.backward(rows(G).to(dev()), grads)
    if self_attn:
        d_t = d_t + d_s
    names = {id(p): n for n, p in blk.named_parameters()}
    grads = {names[k]: v for k, v in grads.items()}
    assert rel_err(out.cpu().double(), rows(r64['out'])) < 2e-5
    for k, v in r64['state'].items():
        if 'running_' in k:
            assert rel_err(blk.state_dict()[k].cpu().double(), v) < 1e-5, k
    checks = [('d_target', d_t.cpu().double(), rows(r64['d_t']), rows(r32['d_t']).double())]
    if not self_attn:
        checks.append(('d_source', d_s.cpu().double(), rows(r64['d_s']), rows(r32['d_s']).double()))
    assert set(grads) == set(r64['grads'])
    for n, ref_g in r64['grads'].items():
        checks.append((n, grads[n].cpu().double().view_as(ref_g), ref_g, r32['grads'][n].double()))
    bad = []
    for n, ours, ref_g, f32 in checks:
        e, e32 = rel_err(ours, ref_g), rel_err(f32, ref_g)
        if not e < max(1e-4, 5 * e32):
            bad.append((n, e, e32))
    assert not bad, bad


def test_encoder_train_step_matches_oracle_autograd():
    """Training-mode step of the whole base encoder (BatchNorm batch statistics and their gradient; I2P dropout p = 0):
    outputs, running statistics after the step, input gradients and EVERY parameter gradient vs torch autograd through
    the CPU oracle in .train(), evaluated in FLOAT64.  The gradients are badly conditioned: fp32 autograd through the same
    oracle is itself up to 1.4e-2 away from float64 on the attention projections (softmax-window and batch-mean
    differences cancel), and the one known forward deviation of the product -- the dense depth map differs by up to 2e-3 m
    from OpenCV's LUT-based bilateral filter (test_gpu_encoder.py::test_bevwarp_stages_match_oracle), i.e. 1e-4 in the warped
    BEV features -- is amplified the same way (measured: parameter gradients of the P2I block up to 1.4e-2, input
    gradients 2e-3; with exact inputs the block-level test above holds 1e-4 / 5x fp32 autograd).  Bars: 5e-3 on the input
    gradients, 3e-2 on every parameter tensor -- structural errors show up as O(1)."""
    from deepinteraction_b200 import mmri, train
    seed = 1570
    r64, r32 = _oracle_train_step(seed, torch.float64), _oracle_train_step(seed, torch.float32)
    fr, Gs = r64['fr'], r64['Gs']
    enc = mmri.DeepInteractionEncoder(2, 64, 64, 128)
    enc.load_state_dict(r64['state0'], strict=True)
    enc = enc.to(dev()).train()
    d = dev()
    nhwc = lambda t: t.detach().permute(0, 2, 3, 1).contiguous().to(d)
    pm = {k: (v.to(d) if torch.is_tensor(v) else [p.to(d) for p in v]) for k, v in fr['pts_metas'].items()}
    r = train.encoder_train_step(enc, fr['img_feats'].to(d), fr['pts_feats'].to(d), fr['img_metas'], pm,
                                 lambda a, b, c: tuple(nhwc(G) for G in Gs))
    nchw = lambda t: t.permute(0, 3, 1, 2).cpu().double()
    for ours, ref, name in zip(r['outputs'], r64['outs'], ('img', 'pts_conv', 'pts')):
        assert rel_err(nchw(ours), ref) < 1e-4, name
    sd_ref, sd = r64['m'].state_dict(), enc.state_dict()
    for k in sd_ref:
        if 'running_' in k:
            assert rel_err(sd[k].cpu().double(), sd_ref[k]) < 1e-4, k
        elif k.endswith('num_batches_tracked'):
            assert int(sd[k]) == int(sd_ref[k]), k
    bar_in, bar_par = 5e-3, 3e-2
    bad, worst = [], (0.0, None, 0.0)
    for ours, ref, f32, name in zip((r['d_img_feats'], r['d_pts_feats']), r64['d_in'], r32['d_in'], ('d img_feats', 'd pts_feats')):
        e, e32 = rel_err(nchw(ours), ref), rel_err(f32.double(), ref)
        print('%s: %.2e (fp32 autograd %.2e)' % (name, e, e32))
        if not e < bar_in:
            bad.append((name, e, e32))
    for name, ref in r64['grads'].items():
        assert ref is not None and name in r['grads'], name
        ours = r['grads'][name].cpu().double().view_as(ref)
        if name.endswith('out_proj.bn.bias'):
            # analytically zero: the next layer's batch-mean subtraction cancels a per-channel constant
            assert float(ref.abs().max()) < 1e-6 and float(ours.abs().max()) < 1e-3, name
            continue
        e, e32 = rel_err(ours, ref), rel_err(r32['grads'][name].double(), ref)
        worst = max(worst, (e, name, e32))
        if not e < bar_par:
            bad.append((name, e, e32))
    print('train step: %d parameter tensors, worst %s %.2e (fp32 autograd %.2e)' % (len(r['grads']), worst[1], worst[0], worst[2]))
    assert not bad, bad


def _dropout_calls(coors, valid, chunk=2048):
    """Row sets (global pillar indices) in the order oracle.mmri.MMRI_I2P calls the attention: per batch sample, valid pillars,
    chunks of `chunk`."""
    out = []
    for b in range(int(coors[:, 0].max()) + 1):
        idx = ((coors[:, 0] == b) & valid).nonzero().squeeze(1)
        out += [idx[s:s + chunk] for s in range(0, idx.numel(), chunk)]
    return out


def test_i2p_attention_dropout_matches_oracle_with_the_same_mask(monkeypatch):
    """Training-mode attention dropout of MMRI_I2P (nn.MultiheadAttention(dropout=p), encoder_utils.py:223): the product draws its
    mask from a counter-based hash, torch from Philox, so the mask the kernels use (di_i2p_dropout_mask_f32) is injected into the
    oracle's F.dropout; output and all gradients must then agree with autograd, and the keep rate must be 1 - p."""
    import torch.nn.functional as F
    import oracle.mmri as om
    from deepinteraction_b200 import mmri, synth, fold, geom, backward, ops
    from test_gpu_encoder import _cfg1_frame
    seed, pdrop, dseed = 1100, 0.3, 20240917
    torch.manual_seed(seed)
    m = om.MMRI_I2P(64, 64, pdrop)
    synth.randomize_norm_stats(m, seed)
    m.train()
    fr = _cfg1_frame(seed, True)
    g = torch.Generator().manual_seed(seed)
    pts = fr['pts_feats'].clone().requires_grad_(True)
    img = fr['img_feats'].clone().requires_grad_(True)
    B = pts.shape[0]
    G = torch.randn(pts.shape, generator=g)
    d = dev()
    mha = m.learnedAlign
    # dropout form of the fold: out = M2x [s, rho, 0, 0, 0] + b_o with rho = sum_j a_j m_j (the value bias is weighted by it)
    M1, c1, M2x, bo = fold.i2p_fold(mha, split_bias=True)
    pack = (fold.Weight(M1, d), fold.dev(c1, d), fold.dev(M2x, d), fold.dev(bo, d))
    enc = mmri.DeepInteractionEncoder(1, 64, 64, 64)
    pm = enc._canon_pts_metas(fr['pts_metas'], d)
    proj, _ = geom.camera_rows(fr['img_metas'], d)
    nhwc = lambda t: t.detach().permute(0, 2, 3, 1).contiguous().to(d)
    P, T = pm['pillars'].shape[:2]
    # ours: forward (through the module-level helper) and backward with dropout = (p, seed)
    geo = type('G', (), dict(proj=proj, V=1, in_hw=(256, 256)))()
    with backward._precise():
        out = enc.i2p(dict(i2p=pack), nhwc(pts), nhwc(img), pm, geo, dropout=(pdrop, dseed))
    r = backward.i2p_backward(pack, nhwc(pts), nhwc(img), pm, proj, 1, (256, 256), nhwc(G), dropout=(pdrop, dseed))
    mask = ops.i2p_dropout_mask(P, T * 1, pdrop, dseed, d).cpu()
    vals = mask.unique().tolist()
    print('mask values', vals, 'keep rate %.4f' % float((mask > 0).float().mean()))
    assert len(vals) == 2 and vals[0] == 0.0 and abs(vals[1] - 1.0 / (1.0 - pdrop)) < 1e-6
    assert abs(float((mask > 0).float().mean()) - (1 - pdrop)) < 0.01
    # the p = 0 variant of the dropout entry point is the plain kernel
    rows = ops.gather_rows(nhwc(pts), pm['pillar_coors'])
    qk = ops.linear([rows], pack[0], pack[1])
    args = (qk, pm['pillars'], pm['pillars_num_points'], pm['pillar_coors'], proj, nhwc(img), 1, (256, 256))
    s0, cnt = ops.i2p_attend(*args)
    s1, _ = ops.i2p_attend(*args, dropout=(1e-30, 5))
    rho = s1[:, 64]
    print('p -> 0 variant vs plain kernel: %.2e, rho in [%.7f, %.7f]' % (rel_err(s1[:, :64], s0), float(rho[cnt > 0].min()), float(rho.max())))
    assert s1.shape == (P, 68) and rel_err(s1[:, :64], s0) < 1e-6 and float(s1[:, 65:].abs().max()) == 0.0
    assert float((rho[cnt > 0] - 1).abs().max()) < 1e-6 and float(rho[cnt == 0].abs().max()) == 0.0
    # oracle with the same mask
    calls = _dropout_calls(pm['pillar_coors'].cpu().long(), cnt.cpu() > 0)

    def fake_dropout(x, p=0.5, training=True, inplace=False):
        rows_ = calls.pop(0)
        assert abs(p - pdrop) < 1e-12 and training and x.shape[0] == rows_.numel(), (p, x.shape, rows_.numel())
        return x * mask[rows_].view(x.shape).to(x.dtype)
    monkeypatch.setattr(F, 'dropout', fake_dropout)
    with torch.enable_grad():
        ref = m(pts, img.view(B, 1, *img.shape[1:]), fr['img_metas'], fr['pts_metas'])
        (ref * G).sum().backward()
    assert not calls
    tol = 1e-4
    e_out = rel_err(out.permute(0, 3, 1, 2).cpu(), ref.detach())
    e_pts, e_img = rel_err(r['d_pts'].permute(0, 3, 1, 2).cpu(), pts.grad), rel_err(r['d_img'].permute(0, 3, 1, 2).cpu(), img.grad)
    print('dropout step vs oracle with the same mask: out %.2e, d_pts %.2e, d_img %.2e' % (e_out, e_pts, e_img))
    assert e_out < tol and e_pts < tol and e_img < tol
    pg = fold.i2p_unfold_grads(mha, r['dM1'], r['dc1'], r['dM2'], r['dc2'])
    Wq_g, Wk_g, Wv_g = (mha.in_proj_weight.grad.chunk(3, 0) if mha._qkv_same_embed_dim else
                        (mha.q_proj_weight.grad, mha.k_proj_weight.grad, mha.v_proj_weight.grad))
    bq_g, _, bv_g = mha.in_proj_bias.grad.chunk(3, 0)
    for name, want in (('Wq', Wq_g), ('Wk', Wk_g), ('Wv', Wv_g), ('bq', bq_g), ('bv', bv_g),
                       ('Wo', mha.out_proj.weight.grad), ('bo', mha.out_proj.bias.grad)):
        assert rel_err(pg[name].float(), want) < tol, name
