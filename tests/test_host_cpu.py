"""CPU: host-side logic of the product path (weight folding, geometry folding, plug-in registry / config
loading, state-dict schema, sharding over a 2-rank gloo group).  No kernel launches."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_err
from tools.ref_goldens import REF_CONFIGS, ref_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUR_CFG = os.path.join(ROOT, 'projects', 'configs', 'nuscenes', 'di_b200_base_hotpath.py')


def load_cfg(src):
    """A config file of this repository, or a reference config by name (its plug-in part, tests/golden/ref_configs.pt)."""
    from projects.mmdet3d_plugin.registry import load_config
    if src in REF_CONFIGS:
        return ref_config(src)
    return load_config(src if os.path.isabs(src) else os.path.join(ROOT, src))


def test_conv_bn_and_fuse_pair_folding():
    import oracle.mmri as om
    from deepinteraction_b200 import fold, synth, mmri
    torch.manual_seed(0)
    C = 16
    a, b = om.ConvBNReLU(2 * C, C, 1, act=False).eval(), om.ConvBNReLU(2 * C, C, 1, act=False).eval()
    synth.randomize_norm_stats(a, 1)
    synth.randomize_norm_stats(b, 2)
    x, y, z = (torch.randn(3, C, 5, 7) for _ in range(3))
    with torch.no_grad():
        ref = b(torch.cat((a(torch.cat((x, y), 1)), z), 1))
    ha, hb = mmri.ConvBN(2 * C, C), mmri.ConvBN(2 * C, C)
    ha.load_state_dict(a.state_dict())
    hb.load_state_dict(b.state_dict())
    W, bias = fold.fuse_pair(ha, hb)
    rows = torch.cat([t.permute(0, 2, 3, 1).reshape(-1, C) for t in (x, y, z)], 1).double()
    out = (rows @ W.t() + bias).float().view(3, 5, 7, C).permute(0, 3, 1, 2)
    assert rel_err(out, ref) < 1e-5


def test_i2p_attention_fold_equals_multihead_attention():
    from deepinteraction_b200 import fold
    torch.manual_seed(1)
    C = 32
    mha = torch.nn.MultiheadAttention(C, 1, kdim=C, vdim=C, batch_first=True).eval()
    with torch.no_grad():
        mha.in_proj_bias.normal_(0, 0.1)
        mha.out_proj.bias.normal_(0, 0.1)
    q, kv = torch.randn(7, 1, C), torch.randn(7, 11, C)
    mask = torch.rand(7, 1, 11) > 0.6
    mask[:, :, 0] = False
    with torch.no_grad():
        ref = mha(q, kv, kv, attn_mask=mask)[0][:, 0]
    M1, c1, M2, c2 = fold.i2p_fold(mha)
    qk = q[:, 0].double() @ M1.t() + c1
    logits = torch.einsum('pc,pkc->pk', qk, kv.double()).masked_fill(mask[:, 0], float('-inf'))
    s = torch.einsum('pk,pkc->pc', logits.softmax(-1), kv.double())
    out = (s @ M2.t() + c2).float()
    assert rel_err(out, ref) < 1e-5


def test_i2p_unfold_grads_is_the_chain_rule_of_the_fold():
    """fold.i2p_unfold_grads maps gradients w.r.t. the folded (M1, c1, M2, c2) back to nn.MultiheadAttention's own parameters:
    compared with autograd through the module itself (the training step relies on it, train.py)."""
    from deepinteraction_b200 import fold
    torch.manual_seed(2)
    C = 16
    mha = torch.nn.MultiheadAttention(C, 1, kdim=C, vdim=C, batch_first=True).double()
    with torch.no_grad():
        mha.in_proj_bias.normal_(0, 0.1)
        mha.out_proj.bias.normal_(0, 0.1)
    q, kv, G = torch.randn(9, 1, C).double(), torch.randn(9, 6, C).double(), torch.randn(9, C).double()
    (mha(q, kv, kv)[0][:, 0] * G).sum().backward()
    M1, c1, M2, c2 = (t.clone().requires_grad_(True) for t in fold.i2p_fold(mha))
    qk = q[:, 0] @ M1.t() + c1
    s_ = torch.einsum('pk,pkc->pc', torch.einsum('pc,pkc->pk', qk, kv).softmax(-1), kv)
    ((s_ @ M2.t() + c2) * G).sum().backward()
    u = fold.i2p_unfold_grads(mha, M1.grad, c1.grad, M2.grad, c2.grad)
    W = torch.cat([u['Wq'], u['Wk'], u['Wv']], 0)
    b = torch.cat([u['bq'], u['bk'], u['bv']], 0)
    assert rel_err(W, mha.in_proj_weight.grad) < 1e-10 and rel_err(b, mha.in_proj_bias.grad) < 1e-10
    assert rel_err(u['Wo'], mha.out_proj.weight.grad) < 1e-10 and rel_err(u['bo'], mha.out_proj.bias.grad) < 1e-10
    with fold.on_device():                     # the device-resident variant computes the same thing (CPU tensors here)
        u2 = fold.i2p_unfold_grads(mha, M1.grad, c1.grad, M2.grad, c2.grad)
    assert all(torch.equal(u[k], u2[k]) for k in u)


def test_i2p_fold_with_attention_dropout(monkeypatch):
    """Dropout multiplies the softmax weights by m_j / (1 - p) AFTER normalisation, so they no longer sum to 1 and the value
    bias is weighted by rho = sum_j a_j m_j: fold.i2p_fold(split_bias=True) / i2p_unfold_grads against nn.MultiheadAttention in
    training mode with the same mask injected into F.dropout (forward and every parameter gradient, float64)."""
    import torch.nn.functional as F
    from deepinteraction_b200 import fold
    torch.manual_seed(5)
    C, P, S, pd = 16, 9, 6, 0.3
    mha = torch.nn.MultiheadAttention(C, 1, dropout=pd, kdim=C, vdim=C, batch_first=True).double().train()
    with torch.no_grad():
        mha.in_proj_bias.normal_(0, 0.3)
        mha.out_proj.bias.normal_(0, 0.3)
    q, kv, G = torch.randn(P, 1, C).double(), torch.randn(P, S, C).double(), torch.randn(P, C).double()
    mask = (torch.rand(P, S) >= pd).double() / (1 - pd)
    monkeypatch.setattr(F, 'dropout', lambda x, p=0.5, training=True, inplace=False: x * mask.view(x.shape))
    ref = mha(q, kv, kv)[0][:, 0]
    (ref * G).sum().backward()
    monkeypatch.undo()
    M1, c1, M2x, bo = (t.clone().requires_grad_(True) for t in fold.i2p_fold(mha, split_bias=True))
    assert M2x.shape == (C, C + 4)
    a = torch.einsum('pc,pkc->pk', q[:, 0] @ M1.t() + c1, kv).softmax(-1) * mask
    s_ext = torch.cat([torch.einsum('pk,pkc->pc', a, kv), a.sum(1, keepdim=True), torch.zeros(P, 3).double()], 1)
    out = s_ext @ M2x.t() + bo
    assert rel_err(out.detach(), ref.detach()) < 1e-12
    (out * G).sum().backward()
    u = fold.i2p_unfold_grads(mha, M1.grad, c1.grad, M2x.grad, bo.grad)
    W, b = torch.cat([u['Wq'], u['Wk'], u['Wv']], 0), torch.cat([u['bq'], u['bk'], u['bv']], 0)
    assert rel_err(W, mha.in_proj_weight.grad) < 1e-10 and rel_err(b, mha.in_proj_bias.grad) < 1e-10
    assert rel_err(u['Wo'], mha.out_proj.weight.grad) < 1e-10 and rel_err(u['bo'], mha.out_proj.bias.grad) < 1e-10


def test_grad_sink_reports_gradients_in_backward_order_to_the_buckets():
    """train.GradSink hands every parameter gradient to the callback when it is produced (so shard.GradBuckets can launch full
    buckets during the backward) and keeps the contiguous tensor the buckets later overwrite with the averaged result."""
    from deepinteraction_b200.shard import GradBuckets
    from deepinteraction_b200.train import GradSink
    ps = [torch.nn.Parameter(torch.zeros(3, 2)), torch.nn.Parameter(torch.zeros(5)), torch.nn.Parameter(torch.zeros(2, 2))]
    names = {id(p): 'p%d' % i for i, p in enumerate(ps)}
    buckets, order = GradBuckets(bucket_bytes=32), []
    sink = GradSink(names, lambda n, t: (order.append(n), buckets.add(t)))
    sink[id(ps[2])] = torch.full((2, 2), 2.0)
    sink[id(ps[0])] = torch.arange(6.0).view(2, 3).t()              # a non-contiguous gradient is stored contiguous
    assert buckets.launched == 1                                    # 16 + 24 bytes >= 32: launched before the last gradient exists
    sink[id(ps[1])] = torch.ones(5)
    buckets.finish()
    assert order == ['p2', 'p0', 'p1'] and buckets.launched == 2
    assert all(t.is_contiguous() for t in sink.values())
    assert torch.equal(sink[id(ps[0])], torch.arange(6.0).view(2, 3).t()) and torch.equal(sink[id(ps[1])], torch.ones(5))


def test_lazy_weight_equals_eager_weight():
    from deepinteraction_b200 import fold
    w = torch.randn(24, 40, generator=torch.Generator().manual_seed(3))
    a, b = fold.Weight(w, 'cpu'), fold.Weight(w, 'cpu', lazy=True)
    assert b._tf32 is None and b._bf16 is None
    for k in ('w', 'hi', 'lo', 'bh', 'bm', 'wt'):
        assert torch.equal(getattr(a, k), getattr(b, k)), k
    assert torch.equal(a.hi + a.lo, w) and a.shape == b.shape == (24, 40)


def test_train_mode_batchnorm_formulas():
    """The closed forms csrc/bn_train.cu implements (shifted one-pass block moments merged with Chan's formula; dy = gamma rstd
    (g - mean(g) - xhat mean(g xhat))) against torch.nn.functional.batch_norm + autograd, in float64 on the host."""
    import torch.nn.functional as F
    g_ = torch.Generator().manual_seed(4)
    M, C, eps = 203, 5, 1e-5
    y = (torch.randn(M, C, generator=g_) * 0.3 + torch.tensor([100.0, -3.0, 0.0, 7.0, 0.5])).double()
    parts = []
    for m0 in range(0, M, 37):                                    # row blocks as the kernel forms them
        blk = y[m0:m0 + 37]
        d = blk - blk[0]
        s1, s2, n = d.sum(0), (d * d).sum(0), blk.shape[0]
        parts.append((n, blk[0] + s1 / n, s2 - s1 * s1 / n))
    n, mu, m2 = 0, torch.zeros(C).double(), torch.zeros(C).double()
    for nb, mub, m2b in parts:
        d = mub - mu
        mu, m2, n = mu + d * nb / (n + nb), m2 + m2b + d * d * n * nb / (n + nb), n + nb
    assert rel_err(mu, y.mean(0)) < 1e-12 and rel_err(m2 / M, y.var(0, unbiased=False)) < 1e-10
    gamma, beta, dz = torch.rand(C).double() + 0.5, torch.randn(C).double(), torch.randn(M, C, generator=g_).double()
    yr, gr = y.clone().requires_grad_(True), gamma.clone().requires_grad_(True)
    z = F.relu(F.batch_norm(yr, None, None, gr, beta, True, 0.1, eps))
    (z * dz).sum().backward()
    rstd = 1 / torch.sqrt(m2 / M + eps)
    xhat = (y - mu) * rstd
    g = dz * (z.detach() > 0)
    dy = gamma * rstd * (g - g.mean(0) - xhat * (g * xhat).mean(0))
    assert rel_err(dy, yr.grad) < 1e-9 and rel_err((g * xhat).sum(0), gr.grad) < 1e-10


def test_aug_affine_matches_apply_3d_transformation():
    from oracle.geometry import apply_3d_transformation
    from deepinteraction_b200 import geom, synth
    meta = dict(synth.AUG_META)
    pts = torch.randn(50, 3, dtype=torch.float64) * 20
    for reverse in (False, True):
        ref = apply_3d_transformation(pts, meta, reverse=reverse)
        A = torch.from_numpy(geom.aug_affine(meta, reverse))
        out = (torch.cat([pts, torch.ones(50, 1, dtype=torch.float64)], 1) @ A.t())[:, :3]
        assert float((out - ref).abs().max()) < 1e-9
    assert np.allclose(geom.aug_affine({}, True), np.eye(4))
    # vertical flip and an identity flow entry
    meta2 = dict(pcd_vertical_flip=True, transformation_3d_flow=['VF', 'HF'])
    ref = apply_3d_transformation(pts, meta2, reverse=False)
    out = (torch.cat([pts, torch.ones(50, 1, dtype=torch.float64)], 1) @ torch.from_numpy(geom.aug_affine(meta2, False)).t())[:, :3]
    assert float((out - ref).abs().max()) < 1e-12


def test_camera_rows_project_like_the_oracle():
    import oracle.mmri as om
    from deepinteraction_b200 import geom, synth
    fr = synth.make_frame_batch(7, batch=1, num_views=3, in_hw=(112, 200), n_points=500, aug=True, c_img=4, c_pts=4,
                                bev_hw=(8, 8))
    proj, i2l = geom.camera_rows(fr['img_metas'], 'cpu')
    from oracle.geometry import apply_3d_transformation
    pts = fr['pts_metas']['pts'][0][:, :3]
    p3 = apply_3d_transformation(pts, fr['img_metas'][0], reverse=True)
    l2i = torch.from_numpy(np.asarray(fr['img_metas'][0]['lidar2img']))
    uv, z, mask, _ = om.project_points(p3, l2i, (112, 200))
    cam = torch.einsum('vrk,nk->vnr', proj[0].view(3, 3, 4), torch.cat([pts, torch.ones(len(pts), 1)], 1))
    assert float((cam[..., 2] - z).abs().max()) < 1e-3
    vis = mask
    u2 = cam[..., 0] / cam[..., 2].clamp_min(1e-5)
    assert float((u2 - uv[..., 0])[vis].abs().max()) < 2e-2


@pytest.mark.parametrize('cfg_src', [OUR_CFG, 'Fusion_0075_refactor'])
def test_plugin_builds_from_config_with_reference_state_dict_schema(cfg_src):
    import projects.mmdet3d_plugin  # noqa: F401
    from projects.mmdet3d_plugin.registry import build_hot_path, NECKS, HEADS, BBOX_CODERS
    import oracle.mmri as om
    import oracle.mmpi as omp
    cfg = load_cfg(cfg_src)
    assert cfg['plugin'] is True and cfg['plugin_dir'] == 'projects/mmdet3d_plugin/'
    neck, head = build_hot_path(cfg)
    assert type(neck).__name__ == 'DeepInteractionEncoder' and type(head).__name__ == 'DeepInteractionDecoder'
    m = cfg['model']
    o_neck = om.DeepInteractionEncoder(**{k: v for k, v in m['imgpts_neck'].items() if k != 'type'})
    o_head = omp.DeepInteractionDecoder(test_cfg=m['test_cfg']['pts'],
                                        **{k: v for k, v in m['pts_bbox_head'].items() if k != 'type'})
    # the oracle's state_dict was loaded strictly into the REFERENCE classes by tools/make_goldens.py
    for ours, ref in ((neck, o_neck), (head, o_head)):
        a, b = ours.state_dict(), ref.state_dict()
        assert set(a) == set(b), set(a) ^ set(b)
        for k in a:
            assert a[k].shape == b[k].shape, k
        ours.load_state_dict(b, strict=True)
    assert sum(p.numel() for p in neck.parameters()) == 1780480          # SURVEY.md 8(c): 1.78 M / 21.92 M
    assert sum(p.numel() for p in head.parameters()) == 21922936
    for reg, name in ((NECKS, 'DeepInteractionEncoder'), (HEADS, 'DeepInteractionDecoder'),
                      (BBOX_CODERS, 'TransFusionBBoxCoder')):
        assert reg.get(name) is not None


def test_plusplus_config_builds_its_neck_with_the_reference_schema():
    """The reference's unchanged Fusion_0075_plusplus.py (as stored in tests/golden/ref_configs.pt) builds `imgpts_neck`
    (FusionTransformerv4 + DeepInteractionLayer + MMRI_P2I / MMRI_I2P / MMRI_I2P_Polar) through the plug-in registries;
    state_dict keys and shapes equal the oracle's, whose state_dict tools/make_goldens_pp.py loads strictly into the
    reference classes."""
    import projects.mmdet3d_plugin  # noqa: F401
    from projects.mmdet3d_plugin.registry import build_neck, NECKS, TRANSFORMER_LAYER, ATTENTION
    import oracle.mmri_pp as opp
    cfg = load_cfg('Fusion_0075_plusplus')
    neck = build_neck(cfg)
    assert type(neck).__name__ == 'FusionTransformerv4'
    o = opp.FusionTransformerv4(**{k: v for k, v in cfg['model']['imgpts_neck'].items() if k != 'type'})
    a, b = neck.state_dict(), o.state_dict()
    assert set(a) == set(b), sorted(set(a) ^ set(b))[:8]
    for k in a:
        assert a[k].shape == b[k].shape, k
    neck.load_state_dict(b, strict=True)
    for reg, names in ((NECKS, ['FusionTransformerv4']), (TRANSFORMER_LAYER, ['DeepInteractionLayer']),
                       (ATTENTION, ['MMRI_P2I', 'MMRI_I2P', 'MMRI_I2P_Polar'])):
        for n in names:
            assert reg.get(n) is not None, n


@pytest.mark.parametrize('cfg_src', ['Fusion_0075_plusplus', 'projects/configs/nuscenes/di_b200_plusplus_hotpath.py'])
def test_plusplus_config_builds_its_head_with_the_reference_schema(cfg_src):
    """`pts_bbox_head` of the ++ config (DeepInteractionPlusPlusDecoder: V2 RCNN blocks with ffn / self_ffn / self_norm /
    scale / self_scale, prediction heads on C channels) builds through HEADS; state_dict keys and shapes equal the
    oracle's, whose state_dict tools/make_goldens.py (G7) loads strictly into the reference class."""
    import projects.mmdet3d_plugin  # noqa: F401
    from projects.mmdet3d_plugin.registry import build_hot_path, HEADS
    import oracle.mmpi_pp as opp
    cfg = load_cfg(cfg_src)
    neck, head = build_hot_path(cfg)
    assert type(neck).__name__ == 'FusionTransformerv4' and type(head).__name__ == 'DeepInteractionPlusPlusDecoder'
    assert HEADS.get('DeepInteractionPlusPlusDecoder') is not None
    hc = {k: v for k, v in cfg['model']['pts_bbox_head'].items() if k not in ('type', 'train_cfg')}
    o = opp.DeepInteractionPlusPlusDecoder(test_cfg=cfg['model']['test_cfg']['pts'], **hc)
    a, b = head.state_dict(), o.state_dict()
    assert set(a) == set(b), sorted(set(a) ^ set(b))[:8]
    for k in a:
        assert a[k].shape == b[k].shape, k
    head.load_state_dict(b, strict=True)
    assert any(k.endswith('self_ffn.layers.0.0.weight') for k in a) and 'decode_head.1.self_norm_pts.weight' in a
    assert a['pred_head.0.center.0.conv.weight'].shape[1] == 128          # C, not 2C (:140)


def test_assigner_and_cost_names_are_registered():
    """SURVEY.md 8(b): HungarianAssigner3D / HeuristicAssigner3D (BBOX_ASSIGNERS) and BBox3DL1Cost / BBoxBEVL1Cost /
    IoU3DCost (MATCH_COST) resolve, and the reference's train_cfg.pts.assigner builds with its own kwargs."""
    import projects.mmdet3d_plugin  # noqa: F401
    from projects.mmdet3d_plugin.registry import BBOX_ASSIGNERS, MATCH_COST
    for n in ('HungarianAssigner3D', 'HeuristicAssigner3D'):
        assert BBOX_ASSIGNERS.get(n) is not None, n
    for n in ('BBox3DL1Cost', 'BBoxBEVL1Cost', 'IoU3DCost'):
        assert MATCH_COST.get(n) is not None, n
    a = BBOX_ASSIGNERS.build(dict(type='HungarianAssigner3D', iou_calculator=dict(type='BboxOverlaps3D', coordinate='lidar'),
                                  cls_cost=dict(type='FocalLossCost', gamma=2, alpha=0.25, weight=0.15),
                                  reg_cost=dict(type='BBoxBEVL1Cost', weight=0.25), iou_cost=dict(type='IoU3DCost', weight=0.25)))
    assert (a.cls_cost.weight, a.reg_cost.weight, a.reg_cost.kind, a.iou_cost.weight) == (0.15, 0.25, 0, 0.25)
    from projects.mmdet3d_plugin.registry import build_hot_path
    _, head = build_hot_path(load_cfg('Fusion_0075_refactor'))
    assert type(head.bbox_assigner).__name__ == 'HungarianAssigner3D' and head.train_cfg['pos_weight'] == -1


def test_product_modules_refuse_cpu_and_training():
    from deepinteraction_b200 import mmri
    enc = mmri.DeepInteractionEncoder(1, 8, 8, 16).eval()
    with pytest.raises(RuntimeError, match='CUDA only'):
        enc.pack()


def test_frame_slices_cover_the_batch():
    from deepinteraction_b200.shard import frame_slice
    for total in (1, 7, 16, 17):
        for world in (1, 2, 3, 8):
            seen = []
            for r in range(world):
                s = frame_slice(total, world, r)
                seen += list(range(s.start, s.stop))
            assert seen == list(range(total))


def _gloo_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        import oracle.mmri as om
        from deepinteraction_b200 import synth
        from deepinteraction_b200.shard import frame_slice, gather_frames, max_over_ranks
        torch.manual_seed(5)
        m = om.LocalContextAttentionBlock(16, 16, 9).eval()
        synth.randomize_norm_stats(m, 5)
        g = torch.Generator().manual_seed(6)
        x = torch.randn(5, 16, 9, 11, generator=g)             # 5 frames over 2 ranks: 3 + 2
        sl = frame_slice(5, world, rank)
        with torch.no_grad():
            local = m(x[sl], x[sl])
            full = m(x, x)
        got = gather_frames(local, 5)
        t = max_over_ranks(10.0 + rank)
        ret[rank] = (bool(torch.equal(got, full)), t)
    finally:
        dist.destroy_process_group()


def test_two_rank_gloo_sharding_is_bitwise_equal_to_single_rank():
    import torch.multiprocessing as mp
    import socket
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_gloo_worker, args=(2, port, ret), nprocs=2, join=True)
    assert ret[0][0] and ret[1][0], 'sharded frames must equal the single-process result bit for bit'
    assert ret[0][1] == 11.0 and ret[1][1] == 11.0


def _grad_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        import oracle.mmri as om
        from deepinteraction_b200.shard import GradBuckets, frame_slice
        torch.manual_seed(5)
        m = om.LocalContextAttentionBlock(16, 16, 9).eval()
        g = torch.Generator().manual_seed(6)
        x = torch.randn(4, 16, 9, 11, generator=g)
        tgt = torch.randn(4, 16, 9, 11, generator=g)
        # data-parallel step: every rank takes its frames, local sum-of-squares loss, bucketed all-reduce of the gradients
        sl = frame_slice(4, world, rank)
        with torch.enable_grad():
            ((m(x[sl], x[sl]) - tgt[sl]) ** 2).sum().backward()
        buckets = GradBuckets(bucket_bytes=2048)               # small buckets: several launches during the "backward"
        from deepinteraction_b200.train import GradSink          # the training step's gradient store feeds the buckets
        params = [p for p in m.parameters() if p.grad is not None]
        sink = GradSink({id(p): str(i) for i, p in enumerate(params)}, lambda n, t: buckets.add(t))
        for p in reversed(params):                              # the order a backward pass produces them
            sink[id(p)] = p.grad
        buckets.finish()
        grads = [sink[id(p)] for p in params]                   # overwritten in place with the rank average
        # single-process reference over all frames (averaged over ranks, as DDP does)
        ref = om.LocalContextAttentionBlock(16, 16, 9).eval()
        ref.load_state_dict(m.state_dict())
        with torch.enable_grad():
            ((ref(x, x) - tgt) ** 2).sum().backward()
        want = [p.grad / world for p in ref.parameters() if p.grad is not None]
        err = max(float((a - b).abs().max() / b.abs().max().clamp_min(1e-12)) for a, b in zip(grads, want))
        ret[rank] = (err, buckets.launched, [float(gr.sum()) for gr in grads])
    finally:
        dist.destroy_process_group()


def test_two_rank_gloo_bucketed_gradient_allreduce():
    """SURVEY.md 8(e): the training path's one collective -- bucketed gradient all-reduce -- on 2 gloo ranks: averaged
    gradients equal the single-process gradients of the whole batch / world, identical on both ranks, several buckets."""
    import torch.multiprocessing as mp
    import socket
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    ret = mp.Manager().dict()
    mp.spawn(_grad_worker, args=(2, port, ret), nprocs=2, join=True)
    assert ret[0][0] < 1e-5 and ret[1][0] < 1e-5, (ret[0][0], ret[1][0])
    assert ret[0][1] > 1 and ret[0][2] == ret[1][2]


def test_presplit_operand_format_roundtrip():
    """fold.split_rows = host model of the window kernel's pre-split operand format (gemm_tc.cu split_block)."""
    from deepinteraction_b200 import fold
    g = torch.Generator().manual_seed(0)
    x = torch.randn(37, 64, generator=g) * torch.logspace(-3, 3, 64)
    for kind in (1, 2):
        w = fold.split_rows(x, kind).view(torch.int32)
        if kind == 1:
            wh, wm = w[:, 0::2], w[:, 1::2]
        else:
            v = w.view(37, 8, 8)
            wh, wm = v[:, :, :4].reshape(37, 32), v[:, :, 4:].reshape(37, 32)
        unpack = lambda t: torch.stack([(t << 16), (t & -65536)], -1).view(torch.float32).reshape(37, 64)
        rec = unpack(wh) + unpack(wm)
        assert float(((rec - x).abs() / x.abs()).max()) <= 2.0 ** -16
    # kind 3 (planar, tcgen05 window kernel): 128 channels -> 64 hi words | 64 mid words
    x3 = torch.randn(37, 256, generator=g) * torch.logspace(-3, 3, 256)
    w = fold.split_rows(x3, 3).view(torch.int32).view(37, 2, 128)
    wh, wm = w[:, :, :64].reshape(37, 128), w[:, :, 64:].reshape(37, 128)
    unpack = lambda t: torch.stack([(t << 16), (t & -65536)], -1).view(torch.float32).reshape(37, 256)
    assert float((((unpack(wh) + unpack(wm)) - x3).abs() / x3.abs()).max()) <= 2.0 ** -16
